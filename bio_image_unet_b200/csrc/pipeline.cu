// HBM-bound kernels either side of the network: intensity histogram, percentile-normalisation LUT,
// LUT application, tile gather and the three overlap stitches. All integer / byte work is bit-exact
// with the reference's numpy code (citations per kernel).
#include "common.cuh"
#include "launch.h"

namespace biu {

// ------------------------------------------------------------------------------------------------
// Histogram of integer intensities, one 65536-bin table per frame (uint8 input uses bins 0..255).
// Feeds np.percentile / np.min / np.max of unet/predict.py:125-128 without sorting.
// Per-block privatised sub-histogram in shared memory for the low 16K bins (where microscopy data
// lives), global atomics for the rest; 128-bit loads.
// ------------------------------------------------------------------------------------------------
constexpr int kHistBins = 65536;
constexpr int kSmemBins = 8192;

template <typename T>
__global__ void __launch_bounds__(512) histogram_kernel(const T* __restrict__ img, long long n_per_frame,
                                                         unsigned int* __restrict__ hist, int blocks_per_frame) {
  __shared__ unsigned int sh[kSmemBins];
  const int frame = blockIdx.x / blocks_per_frame;
  const int blk = blockIdx.x % blocks_per_frame;
  for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x) sh[i] = 0;
  __syncthreads();
  const T* src = img + (long long)frame * n_per_frame;
  unsigned int* h = hist + (long long)frame * kHistBins;
  constexpr int VEC = 16 / sizeof(T);
  const long long nvec = n_per_frame / VEC;
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) & 15) == 0);
  if (aligned) {
    const uint4* v = reinterpret_cast<const uint4*>(src);
    for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < nvec; i += (long long)blocks_per_frame * blockDim.x) {
      uint4 q = __ldg(v + i);
      const T* e = reinterpret_cast<const T*>(&q);
#pragma unroll
      for (int k = 0; k < VEC; ++k) {
        const unsigned int b = e[k];
        if (b < kSmemBins) atomicAdd(&sh[b], 1u); else atomicAdd(&h[b], 1u);
      }
    }
    for (long long i = nvec * VEC + (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame;
         i += (long long)blocks_per_frame * blockDim.x) {
      const unsigned int b = src[i];
      if (b < kSmemBins) atomicAdd(&sh[b], 1u); else atomicAdd(&h[b], 1u);
    }
  } else {
    for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame;
         i += (long long)blocks_per_frame * blockDim.x) {
      const unsigned int b = src[i];
      if (b < kSmemBins) atomicAdd(&sh[b], 1u); else atomicAdd(&h[b], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < kSmemBins; i += blockDim.x)
    if (sh[i]) atomicAdd(&h[i], sh[i]);
}

int launch_histogram(const void* img, int dtype_bytes, long long n_per_frame, int frames, unsigned int* hist,
                     cudaStream_t stream) {
  BIU_REQUIRE(dtype_bytes == 1 || dtype_bytes == 2, "histogram: only uint8/uint16 input (got %d-byte)", dtype_bytes);
  BIU_CHECK_CUDA(cudaMemsetAsync(hist, 0, (size_t)frames * kHistBins * sizeof(unsigned int), stream));
  // a block zeroes and flushes its 8192-bin sub-histogram: give it at least 64 K pixels so that this does not dominate
  long long work = ceil_div_ll(n_per_frame, 512LL * 128);
  int bpf = (int)(work < 1 ? 1 : (work > 592 ? 592 : work));
  if (frames * bpf < 148) bpf = ceil_div(148, frames) < work ? ceil_div(148, frames) : (int)(work < 1 ? 1 : work);
  if (dtype_bytes == 2)
    histogram_kernel<uint16_t><<<frames * bpf, 512, 0, stream>>>((const uint16_t*)img, n_per_frame, hist, bpf);
  else
    histogram_kernel<uint8_t><<<frames * bpf, 512, 0, stream>>>((const uint8_t*)img, n_per_frame, hist, bpf);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

__global__ void hist_sum_kernel(const unsigned int* __restrict__ hist, int frames, unsigned int* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= kHistBins) return;
  unsigned long long s = 0;
  for (int f = 0; f < frames; ++f) s += hist[(long long)f * kHistBins + b];
  // 'all' mode totals can exceed 2^32 pixels only above 4 Gpx per call; the LUT kernel takes 64-bit counts
  // from a 2-word table in that case, not supported here.
  out[b] = (unsigned int)s;
}
int launch_hist_sum(const unsigned int* hist, int frames, unsigned int* out, cudaStream_t stream) {
  hist_sum_kernel<<<kHistBins / 256, 256, 0, stream>>>(hist, frames, out);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Percentile bounds + normalisation look-up table from a histogram, in float64 with numpy's exact
// operation order (no FMA contraction):
//   lo = np.nanpercentile(img, q_lo), hi = np.percentile(img, q_hi)      unet/predict.py:125-126
//   img = clip(img, lo, hi); img = img - min(img); img = img / max(img) * 255; [255 - img]   :125-130
//   stored back with a truncating cast (:131) and cast to uint8 at the split (:175-181).
// np.percentile(method='linear'): virtual index (n-1)*(q/100); a + (b-a)*g, or b - (b-a)*(1-g) when g >= 0.5
// (numpy/lib/_function_base_impl.py _quantile/_lerp).
// One block per frame. params[f] = {lo, hi, mn, mx}.
// ------------------------------------------------------------------------------------------------
__device__ double percentile_from_hist(const unsigned long long* cum_sh, const unsigned int* hist, long long n,
                                       double q) {
  // cum_sh: inclusive prefix counts over 256 coarse groups of 256 bins (shared); fine search inside a group.
  const double quant = __ddiv_rn(q, 100.0);
  const double vi = __dmul_rn((double)(n - 1), quant);
  long long prev = (long long)floor(vi);
  long long next = prev + 1;
  double gamma;
  if (vi >= (double)(n - 1)) {
    prev = n - 1; next = n - 1;
    gamma = __dsub_rn(vi, -1.0);  // numpy subtracts the (already replaced) index -1; the lerp is between equal values
  } else if (vi < 0.0) {
    prev = 0; next = 0;
    gamma = vi;
  } else {
    gamma = __dsub_rn(vi, (double)prev);
  }
  // value of the k-th order statistic = smallest bin v with cumulative count > k
  auto kth = [&](long long k) -> int {
    int g = 0;
    while (g < 255 && (long long)cum_sh[g] <= k) ++g;
    long long c = g == 0 ? 0 : (long long)cum_sh[g - 1];
    int b = g * 256;
    for (; b < g * 256 + 255; ++b) {
      c += hist[b];
      if (c > k) break;
    }
    return b;
  };
  const double a = (double)kth(prev);
  const double b = (double)kth(next);
  const double diff = __dsub_rn(b, a);
  double r = __dadd_rn(a, __dmul_rn(diff, gamma));
  if (gamma >= 0.5) r = __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, gamma)));
  return r;
}

// One order statistic per call site would walk a 256-bin group of the GLOBAL histogram serially (a dependent L2 load per
// step: ~100 us per frame with one block per frame - most of a small job's run time). Here the block scans the
// histogram cooperatively (coalesced), finds the coarse groups of the four order statistics in parallel, stages those
// groups in shared memory for the fine search, and `kLutSplit` blocks per frame each fill one slice of the table
// (every block repeats the cheap parameter computation). The float64 arithmetic and its order are unchanged.
constexpr int kLutSplit = 8;
constexpr int kLutThreads = 1024;

struct OrderStat { long long k; int group; };

__device__ __forceinline__ void percentile_indices(long long n, double q, long long* prev, long long* next, double* gamma) {
  const double quant = __ddiv_rn(q, 100.0);
  const double vi = __dmul_rn((double)(n - 1), quant);
  *prev = (long long)floor(vi);
  *next = *prev + 1;
  if (vi >= (double)(n - 1)) {
    *prev = n - 1; *next = n - 1;
    *gamma = __dsub_rn(vi, -1.0);  // numpy subtracts the (already replaced) index -1; the lerp is between equal values
  } else if (vi < 0.0) {
    *prev = 0; *next = 0;
    *gamma = vi;
  } else {
    *gamma = __dsub_rn(vi, (double)*prev);
  }
}
__device__ __forceinline__ double percentile_lerp(double a, double b, double gamma) {
  const double diff = __dsub_rn(b, a);
  double r = __dadd_rn(a, __dmul_rn(diff, gamma));
  if (gamma >= 0.5) r = __dsub_rn(b, __dmul_rn(diff, __dsub_rn(1.0, gamma)));
  return r;
}

__global__ void __launch_bounds__(kLutThreads) norm_lut_kernel(const unsigned int* __restrict__ hist_bounds,
                                                               const unsigned int* __restrict__ hist_range,
                                                               long long bounds_stride, long long range_stride, double q_lo,
                                                               double q_hi, int invert, uint8_t* __restrict__ lut,
                                                               double* __restrict__ params) {
  __shared__ unsigned long long cum[256];              // inclusive prefix counts over 256 groups of 256 bins
  __shared__ unsigned int fine[4][256];                // the groups holding the four order statistics
  __shared__ long long s_k[4];
  __shared__ int s_g[4], s_val[4];
  __shared__ double s_gamma[2], sp[4];
  __shared__ int s_vmin, s_vmax;
  const int f = blockIdx.x / kLutSplit, part = blockIdx.x % kLutSplit;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const unsigned int* hb = hist_bounds + (long long)f * bounds_stride;
  const unsigned int* hr = hist_range + (long long)f * range_stride;
  if (threadIdx.x == 0) { s_vmin = kHistBins; s_vmax = -1; }
  __syncthreads();
  // group sums (warp w: groups w, w + 32, ...; a lane reads 8 consecutive bins) and the value range of the data
  int lo_b = kHistBins, hi_b = -1;
  for (int g = warp; g < 256; g += kLutThreads / 32) {
    const uint4* pb = reinterpret_cast<const uint4*>(hb + g * 256 + lane * 8);
    const uint4 b0 = __ldg(pb), b1 = __ldg(pb + 1);
    unsigned long long sum = (unsigned long long)b0.x + b0.y + b0.z + b0.w + b1.x + b1.y + b1.z + b1.w;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if (lane == 0) cum[g] = sum;
    const uint4* pr = reinterpret_cast<const uint4*>(hr + g * 256 + lane * 8);
    const uint4 r0 = __ldg(pr), r1 = __ldg(pr + 1);
    const unsigned int rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (rv[i]) { const int bin = g * 256 + lane * 8 + i; lo_b = min(lo_b, bin); hi_b = max(hi_b, bin); }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    lo_b = min(lo_b, __shfl_xor_sync(0xffffffffu, lo_b, o));
    hi_b = max(hi_b, __shfl_xor_sync(0xffffffffu, hi_b, o));
  }
  if (lane == 0 && hi_b >= 0) { atomicMin(&s_vmin, lo_b); atomicMax(&s_vmax, hi_b); }
  __syncthreads();
  if (warp == 0) {                                     // inclusive scan of the 256 group sums: 8 per lane + warp scan
    unsigned long long v[8], run = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) { run += cum[lane * 8 + i]; v[i] = run; }
    unsigned long long incl = run;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    const unsigned long long excl = incl - run;
#pragma unroll
    for (int i = 0; i < 8; ++i) cum[lane * 8 + i] = v[i] + excl;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const long long n = (long long)cum[255];
    percentile_indices(n, q_lo, &s_k[0], &s_k[1], &s_gamma[0]);
    percentile_indices(n, q_hi, &s_k[2], &s_k[3], &s_gamma[1]);
    for (int i = 0; i < 4; ++i) s_g[i] = 255;          // k beyond the data (empty histogram): last group, like the serial walk
  }
  __syncthreads();
  if (threadIdx.x < 256) {                             // the group of order statistic k: first g with cum[g] > k
    const int g = threadIdx.x;
    const long long below = g == 0 ? 0 : (long long)cum[g - 1];
#pragma unroll
    for (int i = 0; i < 4; ++i)
      if ((long long)cum[g] > s_k[i] && below <= s_k[i]) s_g[i] = g;
  }
  __syncthreads();
  fine[threadIdx.x >> 8][threadIdx.x & 255] = __ldg(hb + s_g[threadIdx.x >> 8] * 256 + (threadIdx.x & 255));
  __syncthreads();
  if (threadIdx.x < 4) {                               // smallest bin whose cumulative count exceeds k
    const int i = threadIdx.x, g = s_g[i];
    long long c = g == 0 ? 0 : (long long)cum[g - 1];
    int b = 0;
    for (; b < 255; ++b) {
      c += fine[i][b];
      if (c > s_k[i]) break;
    }
    s_val[i] = g * 256 + b;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const double lo = percentile_lerp((double)s_val[0], (double)s_val[1], s_gamma[0]);
    const double hi = percentile_lerp((double)s_val[2], (double)s_val[3], s_gamma[1]);
    // np.clip = minimum(maximum(x, lo), hi)
    const double cmin = fmin(fmax((double)s_vmin, lo), hi);
    const double cmax = fmin(fmax((double)s_vmax, lo), hi);
    const double mn = cmin;
    const double mx = __dsub_rn(cmax, mn);
    sp[0] = lo; sp[1] = hi; sp[2] = mn; sp[3] = mx;
    if (params && part == 0) { params[f * 4 + 0] = lo; params[f * 4 + 1] = hi; params[f * 4 + 2] = mn; params[f * 4 + 3] = mx; }
  }
  __syncthreads();
  const double lo = sp[0], hi = sp[1], mn = sp[2], mx = sp[3];
  uint8_t* out = lut + (long long)f * kHistBins;
  constexpr int kSlice = kHistBins / kLutSplit;
  for (int v4 = part * kSlice + 4 * threadIdx.x; v4 < (part + 1) * kSlice; v4 += 4 * kLutThreads) {
    uint8_t r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      double x = fmin(fmax((double)(v4 + i), lo), hi);
      x = __dsub_rn(x, mn);
      x = __dmul_rn(__ddiv_rn(x, mx), 255.0);
      if (invert) x = __dsub_rn(255.0, x);
      // truncating float64 -> integer cast; NaN (constant image) -> 0 like the x86 cast numpy performs
      const int q = (x == x) ? (int)x : 0;
      r[i] = (uint8_t)q;
    }
    *reinterpret_cast<uchar4*>(out + v4) = make_uchar4(r[0], r[1], r[2], r[3]);
  }
}

int launch_norm_lut(const unsigned int* hist_bounds, const unsigned int* hist_range, long long bounds_stride,
                    long long range_stride, int frames, double q_lo, double q_hi, int invert, uint8_t* lut,
                    double* params, cudaStream_t stream) {
  norm_lut_kernel<<<frames * kLutSplit, kLutThreads, 0, stream>>>(hist_bounds, hist_range, bounds_stride, range_stride,
                                                                  q_lo, q_hi, invert, lut, params);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// LUT application: uint8 out[i] = lut[frame][img[i]]. 16-byte loads, 8/16-byte stores.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) apply_lut_kernel(const T* __restrict__ img, long long n_per_frame,
                                                         const uint8_t* __restrict__ lut, long long lut_stride,
                                                         uint8_t* __restrict__ out, int blocks_per_frame) {
  // 16 pixels per thread: one (uint8) or two (uint16) 16-byte loads, 16 table look-ups (the table of a frame is 64 KB
  // and stays in L1 / L2), one 16-byte store
  const int frame = blockIdx.x / blocks_per_frame;
  const int blk = blockIdx.x % blocks_per_frame;
  const T* src = img + (long long)frame * n_per_frame;
  uint8_t* dst = out + (long long)frame * n_per_frame;
  const uint8_t* l = lut + (long long)frame * lut_stride;
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) & 15) == 0) && ((reinterpret_cast<uintptr_t>(dst) & 15) == 0);
  const long long nvec = aligned ? n_per_frame / 16 : 0;
  const long long stride = (long long)blocks_per_frame * blockDim.x;
  for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < nvec; i += stride) {
    uint8_t r[16];
    if (sizeof(T) == 2) {
      const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(src) + 2 * i), q1 = __ldg(reinterpret_cast<const uint4*>(src) + 2 * i + 1);
      const unsigned short* e0 = reinterpret_cast<const unsigned short*>(&q0);
      const unsigned short* e1 = reinterpret_cast<const unsigned short*>(&q1);
#pragma unroll
      for (int k = 0; k < 8; ++k) { r[k] = __ldg(l + e0[k]); r[8 + k] = __ldg(l + e1[k]); }
    } else {
      const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(src) + i);
      const uint8_t* e0 = reinterpret_cast<const uint8_t*>(&q0);
#pragma unroll
      for (int k = 0; k < 16; ++k) r[k] = __ldg(l + e0[k]);
    }
    *reinterpret_cast<uint4*>(dst + i * 16) = *reinterpret_cast<uint4*>(r);
  }
  for (long long i = nvec * 16 + (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame; i += stride)
    dst[i] = __ldg(l + src[i]);
}

int launch_apply_lut(const void* img, int dtype_bytes, long long n_per_frame, int frames, const uint8_t* lut,
                     long long lut_stride, uint8_t* out, cudaStream_t stream) {
  BIU_REQUIRE(dtype_bytes == 1 || dtype_bytes == 2, "apply_lut: only uint8/uint16 input");
  long long work = ceil_div_ll(n_per_frame, 256LL * 16 * 2);
  int bpf = (int)(work < 1 ? 1 : (work > 1184 ? 1184 : work));
  if (dtype_bytes == 2)
    apply_lut_kernel<uint16_t><<<frames * bpf, 256, 0, stream>>>((const uint16_t*)img, n_per_frame, lut, lut_stride, out, bpf);
  else
    apply_lut_kernel<uint8_t><<<frames * bpf, 256, 0, stream>>>((const uint8_t*)img, n_per_frame, lut, lut_stride, out, bpf);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Tile gather (unet/predict.py:152-182, siam_unet/predict.py:164-197, unet3d/predict.py:119-153):
// tile n = ((f*nz + iz)*ny + iy)*nx + ix copies src[f, zs[iz]:+pd, ys[iy]:+ph, xs[ix]:+pw]; sources
// smaller than the tile are padded at the far end by reflection (np.pad 'reflect') or zeros ('constant').
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ int reflect_index(int i, int n) {
  if (n == 1) return 0;
  const int period = 2 * (n - 1);
  i %= period;
  if (i < 0) i += period;
  return i < n ? i : period - i;
}

// TSRC = uint8_t: plain copy of an already normalised stack. With a.lut the normalisation is fused in: the source is
// the raw uint8 / uint16 stack and every value goes through the frame's look-up table on its way into the tile (the
// normalised frame is then never written). V pixels per thread (16 when the tile width allows it): runs that lie inside
// the source row and are 16-byte aligned move as whole vectors. Flips of a.xform (test-time augmentation) pick the
// mirrored tile row / plane, and a mirrored x run is loaded as it lies in the source and reversed in registers.
template <typename TSRC, int V>
__global__ void __launch_bounds__(256) gather_tiles_kernel(GatherArgs a) {
  const long long tile_elems = (long long)a.pd * a.ph * a.pw;
  const long long total = (long long)a.F * a.nz * a.ny * a.nx * tile_elems;
  const TSRC* srcb = reinterpret_cast<const TSRC*>(a.src);
  const bool fx = a.xform & XF_FLIP_X, fy = a.xform & XF_FLIP_Y, fz = a.xform & XF_FLIP_Z;
  for (long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * V; idx < total;
       idx += (long long)gridDim.x * blockDim.x * V) {
    long long r = idx;
    const int x = (int)(r % a.pw); r /= a.pw;
    const int y = (int)(r % a.ph); r /= a.ph;
    const int z = (int)(r % a.pd); r /= a.pd;
    const int ix = (int)(r % a.nx); r /= a.nx;
    const int iy = (int)(r % a.ny); r /= a.ny;
    const int iz = (int)(r % a.nz); r /= a.nz;
    const int f = (int)r;
    int sz = a.zs[iz] + (fz ? a.pd - 1 - z : z), sy = a.ys[iy] + (fy ? a.ph - 1 - y : y);
    bool zero = false;
    if (sz >= a.Z) { if (a.pad_mode == 0) sz = reflect_index(sz, a.Z); else zero = true; }
    if (sy >= a.H) { if (a.pad_mode == 0) sy = reflect_index(sy, a.H); else zero = true; }
    const TSRC* row = srcb + (((long long)f * a.Z + sz) * a.H + sy) * a.W;
    const uint8_t* l = a.lut ? a.lut + (long long)f * a.lut_stride : nullptr;
    const int sx0 = a.xs[ix] + (fx ? a.pw - V - x : x);
    TSRC raw[V];
    bool zk[V];
    constexpr bool kVec = (V * sizeof(TSRC)) % 16 == 0;       // whole 16-byte vectors only (V = 4 runs stay scalar)
    if (kVec && !zero && sx0 + V <= a.W && ((reinterpret_cast<uintptr_t>(row + sx0) & 15) == 0)) {
#pragma unroll
      for (int q = 0; q < (int)(V * sizeof(TSRC)) / 16; ++q)
        reinterpret_cast<uint4*>(raw)[q] = __ldg(reinterpret_cast<const uint4*>(row + sx0) + q);
#pragma unroll
      for (int k = 0; k < V; ++k) zk[k] = false;
    } else {
#pragma unroll
      for (int k = 0; k < V; ++k) {
        int sx = sx0 + k;
        zk[k] = zero;
        if (sx >= a.W) { if (a.pad_mode == 0) sx = reflect_index(sx, a.W); else zk[k] = true; }
        raw[k] = zk[k] ? (TSRC)0 : __ldg(row + sx);
      }
    }
    uint8_t v[V];
#pragma unroll
    for (int k = 0; k < V; ++k) v[k] = zk[k] ? (uint8_t)0 : (l ? __ldg(l + raw[k]) : (uint8_t)raw[k]);
    uint32_t* w = reinterpret_cast<uint32_t*>(v);
    if (fx) {                                                  // reverse the V bytes: word order and bytes in a word
      uint32_t rev[V / 4];
#pragma unroll
      for (int q = 0; q < V / 4; ++q) rev[q] = __byte_perm(w[V / 4 - 1 - q], 0, 0x0123);
#pragma unroll
      for (int q = 0; q < V / 4; ++q) w[q] = rev[q];
    }
    if (V == 16) *reinterpret_cast<uint4*>(a.dst + idx) = *reinterpret_cast<uint4*>(v);
    else *reinterpret_cast<uchar4*>(a.dst + idx) = *reinterpret_cast<uchar4*>(v);
  }
}

// Value of tile source pixel (f, sz, sy, sx) after the far-end padding; uint8 tiles go through the table when there is one.
template <typename TSRC, typename TDST>
__device__ __forceinline__ TDST gather_at(const GatherArgs& a, int f, int sz, int sy, int sx) {
  bool zero = false;
  if (sz >= a.Z) { if (a.pad_mode == 0) sz = reflect_index(sz, a.Z); else zero = true; }
  if (sy >= a.H) { if (a.pad_mode == 0) sy = reflect_index(sy, a.H); else zero = true; }
  if (sx >= a.W) { if (a.pad_mode == 0) sx = reflect_index(sx, a.W); else zero = true; }
  if (zero) return (TDST)0;
  const TSRC raw = __ldg(reinterpret_cast<const TSRC*>(a.src) + (((long long)f * a.Z + sz) * a.H + sy) * a.W + sx);
  if constexpr (sizeof(TDST) == 4) {
    return raw;
  } else {
    return a.lut ? __ldg(a.lut + (long long)f * a.lut_stride + raw) : (uint8_t)raw;
  }
}

// Transposed 2D tiles (XF_TRANSPOSE, ph == pw = P, pd == 1): out[i][j] = tile[fy ? P-1-j : j][fx ? P-1-i : i]. A block
// moves 32 x 32 squares: it reads the source square row by row into shared memory and writes it out column by column,
// so that both the global reads and the global writes of a warp are runs of consecutive pixels.
template <typename TSRC, typename TDST>
__global__ void __launch_bounds__(256) gather_tiles_transposed_kernel(GatherArgs a, TDST* __restrict__ dst) {
  __shared__ TDST sh[32][33];
  const int P = a.pw, nsq = (P + 31) / 32;
  const bool fx = a.xform & XF_FLIP_X, fy = a.xform & XF_FLIP_Y;
  const long long total = (long long)a.F * a.nz * a.ny * a.nx * nsq * nsq;
  for (long long sq = blockIdx.x; sq < total; sq += gridDim.x) {
    long long r = sq;
    const int oj0 = (int)(r % nsq) * 32; r /= nsq;
    const int oi0 = (int)(r % nsq) * 32; r /= nsq;
    const long long n = r;
    const int ix = (int)(r % a.nx); r /= a.nx;
    const int iy = (int)(r % a.ny); r /= a.ny;
    const int iz = (int)(r % a.nz); r /= a.nz;
    const int f = (int)r;
    for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {   // sh[rr][c] = out[oi0 + c][oj0 + rr]
      const int i = oi0 + threadIdx.x, j = oj0 + rr;
      if (i < P && j < P)
        sh[rr][threadIdx.x] = gather_at<TSRC, TDST>(a, f, a.zs[iz], a.ys[iy] + (fy ? P - 1 - j : j),
                                                    a.xs[ix] + (fx ? P - 1 - i : i));
    }
    __syncthreads();
    for (int c = threadIdx.y; c < 32; c += blockDim.y) {
      const int i = oi0 + c, j = oj0 + threadIdx.x;
      if (i < P && j < P) dst[n * P * P + (long long)i * P + j] = sh[threadIdx.x][c];
    }
    __syncthreads();
  }
}

template <typename TSRC, typename TDST>
static void launch_gather_transposed(const GatherArgs& a, TDST* dst, cudaStream_t stream) {
  const int nsq = (a.pw + 31) / 32;
  long long blocks = (long long)a.F * a.nz * a.ny * a.nx * nsq * nsq;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  gather_tiles_transposed_kernel<TSRC, TDST><<<(int)blocks, dim3(32, 8), 0, stream>>>(a, dst);
}

static int check_xform(const GatherArgs& a) {
  BIU_REQUIRE(a.xform >= 0 && a.xform <= (XF_FLIP_X | XF_FLIP_Y | XF_FLIP_Z | XF_TRANSPOSE), "gather: bad transform %d",
              a.xform);
  BIU_REQUIRE(!(a.xform & XF_TRANSPOSE) || (a.ph == a.pw && a.pd == 1 && !(a.xform & XF_FLIP_Z)),
              "gather: a transposed tile must be a square 2D tile (got %d x %d x %d)", a.pd, a.ph, a.pw);
  return 0;
}

int launch_gather_tiles(const GatherArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(a.pw % 4 == 0, "gather_tiles: tile width must be a multiple of 4 (got %d)", a.pw);
  BIU_REQUIRE(a.src_bytes == 1 || (a.src_bytes == 2 && a.lut != nullptr),
              "gather_tiles: a uint16 source needs the look-up table of the fused normalisation");
  if (int rc = check_xform(a)) return rc;
  if (a.xform & XF_TRANSPOSE) {
    if (a.src_bytes == 2) launch_gather_transposed<uint16_t, uint8_t>(a, a.dst, stream);
    else launch_gather_transposed<uint8_t, uint8_t>(a, a.dst, stream);
    BIU_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  const int v = (a.pw % 16 == 0) ? 16 : 4;
  const long long total = (long long)a.F * a.nz * a.ny * a.nx * a.pd * a.ph * a.pw / v;
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  if (a.src_bytes == 2) {
    if (v == 16) gather_tiles_kernel<uint16_t, 16><<<(int)blocks, 256, 0, stream>>>(a);
    else gather_tiles_kernel<uint16_t, 4><<<(int)blocks, 256, 0, stream>>>(a);
  } else {
    if (v == 16) gather_tiles_kernel<uint8_t, 16><<<(int)blocks, 256, 0, stream>>>(a);
    else gather_tiles_kernel<uint8_t, 4><<<(int)blocks, 256, 0, stream>>>(a);
  }
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Test-time augmentation merge: pass p of K adds the inverse-transformed output of the net on the transformed tiles
// into the fp32 running sum, acc = ((v_0 + v_1) + ...) in pass order; pass 0 writes acc and the last pass writes
// mean = acc * (1/K) (exact, K is a power of two) as float32 and / or as uint8 with the head epilogue's truncating
// trunc(mean * 255). Gather formulation (every output element is written by one thread), no atomics: deterministic.
// A block handles a 32 x 32 square of one output plane; for a transposed pass the square of val is staged in shared
// memory so that reads and writes are both runs along x.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) tta_accumulate_kernel(TtaAccArgs a) {
  __shared__ float sh[32][33];
  const bool fx = a.xform & XF_FLIP_X, fy = a.xform & XF_FLIP_Y, fz = a.xform & XF_FLIP_Z;
  const bool tr = a.xform & XF_TRANSPOSE;
  const int nsy = (a.ph + 31) / 32, nsx = (a.pw + 31) / 32;
  const long long total = a.planes * a.pd * nsy * nsx;
  const long long plane_elems = (long long)a.ph * a.pw;
  const bool first = a.pass == 0, last = a.pass == a.passes - 1;
  const float inv_k = 1.0f / (float)a.passes;
  for (long long sq = blockIdx.x; sq < total; sq += gridDim.x) {
    long long r = sq;
    const int x0 = (int)(r % nsx) * 32; r /= nsx;
    const int y0 = (int)(r % nsy) * 32; r /= nsy;
    const int z = (int)(r % a.pd); r /= a.pd;
    const long long p = r;
    const long long obase = (p * a.pd + z) * plane_elems;
    const float* vplane = a.val + (p * a.pd + (fz ? a.pd - 1 - z : z)) * plane_elems;
    if (tr) {                                            // out[y][x] = val[fx ? P-1-x : x][fy ? P-1-y : y]
      for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
        const int x = x0 + rr, y = y0 + threadIdx.x;       // sh[rr][c] = out[y0 + c][x0 + rr]
        if (x < a.pw && y < a.ph)
          sh[rr][threadIdx.x] = __ldg(vplane + (long long)(fx ? a.pw - 1 - x : x) * a.pw + (fy ? a.ph - 1 - y : y));
      }
      __syncthreads();
    }
    for (int rr = threadIdx.y; rr < 32; rr += blockDim.y) {
      const int y = y0 + rr, x = x0 + threadIdx.x;
      if (y >= a.ph || x >= a.pw) continue;
      const float v = tr ? sh[threadIdx.x][rr]
                         : __ldg(vplane + (long long)(fy ? a.ph - 1 - y : y) * a.pw + (fx ? a.pw - 1 - x : x));
      const long long o = obase + (long long)y * a.pw + x;
      const float s = first ? v : __fadd_rn(a.acc[o], v);
      if (!last) {
        a.acc[o] = s;
      } else {
        const float m = __fmul_rn(s, inv_k);
        if (a.out_f32) a.out_f32[o] = m;
        if (a.out_u8) a.out_u8[o] = (uint8_t)(m * 255.0f);   // as the head epilogues (unet/predict.py:200)
      }
    }
    if (tr) __syncthreads();
  }
}

int launch_tta_accumulate(const TtaAccArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(a.passes >= 1 && a.pass >= 0 && a.pass < a.passes, "tta_accumulate: pass %d of %d", a.pass, a.passes);
  BIU_REQUIRE((a.passes & (a.passes - 1)) == 0, "tta_accumulate: the pass count must be a power of two (got %d)",
              a.passes);
  BIU_REQUIRE(a.xform >= 0 && a.xform <= (XF_FLIP_X | XF_FLIP_Y | XF_FLIP_Z | XF_TRANSPOSE), "tta_accumulate: bad transform");
  BIU_REQUIRE(!(a.xform & XF_TRANSPOSE) || (a.ph == a.pw && a.pd == 1 && !(a.xform & XF_FLIP_Z)),
              "tta_accumulate: a transposed tile must be a square 2D tile");
  BIU_REQUIRE(a.pass == a.passes - 1 ? (a.out_u8 || a.out_f32) : a.acc != nullptr,
              "tta_accumulate: the last pass needs an output, the others the accumulator");
  const long long total = a.planes * a.pd * ((a.ph + 31) / 32) * ((a.pw + 31) / 32);
  long long blocks = total;
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  tta_accumulate_kernel<<<(int)blocks, dim3(32, 8), 0, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// 2D overlap stitch (unet/predict.py:204-229, siam_unet/predict.py:217-240): nanmean over the tiles
// covering a pixel followed by a truncating uint8 cast == integer sum // count (checked exhaustively
// in tests). Gather formulation: one thread per 4 output pixels, no atomics, deterministic.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stitch_mean_kernel(StitchMeanArgs a) {
  // 16 output pixels per thread; a covering tile contributes a run of up to 16 bytes, loaded as one vector when it
  // lies inside the tile row and is 16-byte aligned (tile starts that are multiples of 16: every default grid)
  const int W16 = (a.W + 15) / 16;
  const long long total = (long long)a.F * a.C * a.H * W16;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int x16 = (int)(r % W16) * 16; r /= W16;
    const int y = (int)(r % a.H); r /= a.H;
    const int c = (int)(r % a.C); r /= a.C;
    const int f = (int)r;
    unsigned int sum[16], cnt[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) { sum[q] = 0; cnt[q] = 0; }
    for (int j = 0; j < a.ny; ++j) {
      const int ty = y - a.ys[j];
      if (ty < 0 || ty >= a.ph) continue;
      for (int k = 0; k < a.nx; ++k) {
        const int tx0 = x16 - a.xs[k];
        if (tx0 <= -16 || tx0 >= a.pw) continue;
        const uint8_t* t = a.tiles + ((((long long)f * a.ny + j) * a.nx + k) * a.C + c) * a.ph * a.pw + (long long)ty * a.pw;
        if (tx0 >= 0 && tx0 + 16 <= a.pw && ((reinterpret_cast<uintptr_t>(t + tx0) & 15) == 0)) {
          const uint4 v4 = __ldg(reinterpret_cast<const uint4*>(t + tx0));
          const uint8_t* e = reinterpret_cast<const uint8_t*>(&v4);
#pragma unroll
          for (int q = 0; q < 16; ++q) { sum[q] += e[q]; cnt[q] += 1; }
        } else {
#pragma unroll
          for (int q = 0; q < 16; ++q) {
            const int tx = tx0 + q;
            if (tx >= 0 && tx < a.pw) { sum[q] += __ldg(t + tx); cnt[q] += 1; }
          }
        }
      }
    }
    uint8_t o16[16];
#pragma unroll
    for (int q = 0; q < 16; ++q)                       // uncovered -> nanmean of nothing = nan -> 0
      o16[q] = cnt[q] ? (uint8_t)(sum[q] / cnt[q]) : (uint8_t)0;
    uint8_t* o = a.out + (((long long)f * a.C + c) * a.H + y) * a.W + x16;
    if (x16 + 16 <= a.W && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      *reinterpret_cast<uint4*>(o) = *reinterpret_cast<uint4*>(o16);
    } else {
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if (x16 + q < a.W) o[q] = o16[q];
    }
  }
}
int launch_stitch_mean(const StitchMeanArgs& a, cudaStream_t stream) {
  const long long total = (long long)a.F * a.C * a.H * ((a.W + 15) / 16);
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  stitch_mean_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// 3D stitch (unet3d/predict.py:173-195): patch n is written into slot n % 3 of a float16 NaN buffer,
// later patches overwrite earlier ones in the same slot; result = trunc(nanmean over the 3 slots).
// Gather formulation: per voxel and slot keep the covering patch with the largest n; mean of <= 3 integers
// evaluated as float16(sum)/count in float16 then truncated (== numpy's float16 nanmean path).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stitch_mod3_kernel(StitchMod3Args a) {
  // 16 consecutive x voxels per thread. Patches are visited in increasing n (z -> y -> x order), so within a slot a
  // later patch simply overwrites an earlier one - exactly the reference's assignment order.
  const int W16 = (a.W + 15) / 16;
  const long long total = (long long)a.Z * a.H * W16;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int x16 = (int)(r % W16) * 16; r /= W16;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)r;
    uint8_t v0[16], v1[16], v2[16];
    unsigned int has0 = 0, has1 = 0, has2 = 0;           // bit q: slot holds a value for voxel q
#pragma unroll
    for (int q = 0; q < 16; ++q) { v0[q] = 0; v1[q] = 0; v2[q] = 0; }
    for (int i = 0; i < a.nz; ++i) {
      const int tz = z - a.zs[i];
      if (tz < 0 || tz >= a.pd) continue;
      for (int j = 0; j < a.ny; ++j) {
        const int ty = y - a.ys[j];
        if (ty < 0 || ty >= a.ph) continue;
        for (int k = 0; k < a.nx; ++k) {
          const int tx0 = x16 - a.xs[k];
          if (tx0 <= -16 || tx0 >= a.pw) continue;
          const int n = (i * a.ny + j) * a.nx + k;
          const uint8_t* t = a.tiles + (((long long)n * a.pd + tz) * a.ph + ty) * a.pw;
          uint8_t e[16];
          unsigned int m = 0;
          if (tx0 >= 0 && tx0 + 16 <= a.pw && ((reinterpret_cast<uintptr_t>(t + tx0) & 15) == 0)) {
            *reinterpret_cast<uint4*>(e) = __ldg(reinterpret_cast<const uint4*>(t + tx0));
            m = 0xffffu;
          } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const int tx = tx0 + q;
              e[q] = 0;
              if (tx >= 0 && tx < a.pw) { e[q] = __ldg(t + tx); m |= 1u << q; }
            }
          }
          const int sl = n % 3;
          if (sl == 0) {
#pragma unroll
            for (int q = 0; q < 16; ++q) if ((m >> q) & 1u) v0[q] = e[q];
            has0 |= m;
          } else if (sl == 1) {
#pragma unroll
            for (int q = 0; q < 16; ++q) if ((m >> q) & 1u) v1[q] = e[q];
            has1 |= m;
          } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) if ((m >> q) & 1u) v2[q] = e[q];
            has2 |= m;
          }
        }
      }
    }
    uint8_t o16[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) {
      const int c0 = (has0 >> q) & 1, c1 = (has1 >> q) & 1, c2 = (has2 >> q) & 1;
      const int cnt = c0 + c1 + c2;
      const int sum = (c0 ? v0[q] : 0) + (c1 ? v1[q] : 0) + (c2 ? v2[q] : 0);
      o16[q] = cnt ? (uint8_t)(sum / cnt) : (uint8_t)0;
    }
    uint8_t* o = a.out + ((long long)z * a.H + y) * a.W + x16;
    if (x16 + 16 <= a.W && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      *reinterpret_cast<uint4*>(o) = *reinterpret_cast<uint4*>(o16);
    } else {
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if (x16 + q < a.W) o[q] = o16[q];
    }
  }
}
int launch_stitch_mod3(const StitchMod3Args& a, cudaStream_t stream) {
  const long long total = (long long)a.Z * a.H * ((a.W + 15) / 16);
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  stitch_mod3_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Weighted overlap stitch (engine-only, no reference counterpart): out = (sum w * v) // (sum w) over the tiles covering
// an element, w = w_d[tz] * w_h[ty] * w_w[tx] (each table entry in [0, 1024], so w <= 2^30 and w * v < 2^38), in exact
// unsigned 64-bit integer arithmetic: the result does not depend on the order of the sum. Gather form of
// stitch_mean_kernel (16 output elements per thread, one 16-byte load per covering tile where aligned, no atomics).
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stitch_weighted_kernel(StitchWeightedArgs a) {
  extern __shared__ unsigned int s_w[];                // [pd] w_d | [ph] w_h | [pw] w_w
  unsigned int* s_wd = s_w;
  unsigned int* s_wh = s_w + a.pd;
  unsigned int* s_ww = s_wh + a.ph;
  for (int i = threadIdx.x; i < a.pd + a.ph + a.pw; i += blockDim.x)
    s_w[i] = (unsigned int)__ldg(i < a.pd ? a.w_d + i : (i < a.pd + a.ph ? a.w_h + (i - a.pd) : a.w_w + (i - a.pd - a.ph)));
  __syncthreads();
  const int W16 = (a.W + 15) / 16;
  const int ntiles = a.nz * a.ny * a.nx;
  const long long total = (long long)a.F * a.C * a.Z * a.H * W16;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int x16 = (int)(r % W16) * 16; r /= W16;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)(r % a.Z); r /= a.Z;
    const int c = (int)(r % a.C); r /= a.C;
    const int f = (int)r;
    unsigned long long num[16], den[16];
#pragma unroll
    for (int q = 0; q < 16; ++q) { num[q] = 0; den[q] = 0; }
    for (int i = 0; i < a.nz; ++i) {
      const int tz = z - a.zs[i];
      if (tz < 0 || tz >= a.pd) continue;
      for (int j = 0; j < a.ny; ++j) {
        const int ty = y - a.ys[j];
        if (ty < 0 || ty >= a.ph) continue;
        const unsigned int wzy = s_wd[tz] * s_wh[ty];   // <= 2^20: the tile row's factor
        for (int k = 0; k < a.nx; ++k) {
          const int tx0 = x16 - a.xs[k];
          if (tx0 <= -16 || tx0 >= a.pw) continue;
          const long long n = (long long)f * ntiles + (i * a.ny + j) * a.nx + k;
          const uint8_t* t = a.tiles + (((n * a.C + c) * a.pd + tz) * a.ph + ty) * a.pw;
          if (tx0 >= 0 && tx0 + 16 <= a.pw && ((reinterpret_cast<uintptr_t>(t + tx0) & 15) == 0)) {
            const uint4 v4 = __ldg(reinterpret_cast<const uint4*>(t + tx0));
            const uint8_t* e = reinterpret_cast<const uint8_t*>(&v4);
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const unsigned int w = wzy * s_ww[tx0 + q];
              num[q] += (unsigned long long)w * e[q];
              den[q] += w;
            }
          } else {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
              const int tx = tx0 + q;
              if (tx >= 0 && tx < a.pw) {
                const unsigned int w = wzy * s_ww[tx];
                num[q] += (unsigned long long)w * __ldg(t + tx);
                den[q] += w;
              }
            }
          }
        }
      }
    }
    uint8_t o16[16];
#pragma unroll
    for (int q = 0; q < 16; ++q)                       // no covering tile, or zero weight: 0
      o16[q] = den[q] ? (uint8_t)(num[q] / den[q]) : (uint8_t)0;
    uint8_t* o = a.out + ((((long long)f * a.C + c) * a.Z + z) * a.H + y) * a.W + x16;
    if (x16 + 16 <= a.W && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      *reinterpret_cast<uint4*>(o) = *reinterpret_cast<uint4*>(o16);
    } else {
#pragma unroll
      for (int q = 0; q < 16; ++q)
        if (x16 + q < a.W) o[q] = o16[q];
    }
  }
}
int launch_stitch_weighted(const StitchWeightedArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(a.tiles && a.out && a.zs && a.ys && a.xs && a.w_d && a.w_h && a.w_w, "stitch_weighted: null pointer");
  BIU_REQUIRE(a.F > 0 && a.C > 0 && a.Z > 0 && a.H > 0 && a.W > 0, "stitch_weighted: bad output extents F=%d C=%d Z=%d H=%d W=%d",
              a.F, a.C, a.Z, a.H, a.W);
  BIU_REQUIRE(a.nz > 0 && a.ny > 0 && a.nx > 0 && a.pd > 0 && a.ph > 0 && a.pw > 0,
              "stitch_weighted: bad grid %dx%dx%d or tile %dx%dx%d", a.nz, a.ny, a.nx, a.pd, a.ph, a.pw);
  const long long table_bytes = 4LL * (a.pd + a.ph + a.pw);
  BIU_REQUIRE(table_bytes <= 48 * 1024, "stitch_weighted: tile extents %d + %d + %d exceed the shared-memory tables",
              a.pd, a.ph, a.pw);
  const long long total = (long long)a.F * a.C * a.Z * a.H * ((a.W + 15) / 16);
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  stitch_weighted_kernel<<<(int)blocks, 256, (size_t)table_bytes, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ------------------------------------------------------------------------------------------------
// Multi-output 3D blend (multi_output_unet3d/predict.py:203-307, blend_margin rules as written):
// weight starts at 1; z rule, then y rule, then x rule overwrite (not multiply); the "far side" ramps all
// land on index 0 with final value (margin-1)/margin. Accumulation order = patch order z -> y -> x in fp32.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ramp_weight(int z, int y, int x, int iz, int iy, int ix, int nz, int ny, int nx,
                                             int margin) {
  float w = 1.0f;
  const int mz = margin < nz ? margin : nz;   // :254 uses min(blend_margin, self.N_z) — patch COUNT, as written
  if (iz > 0 && z < mz) w = (float)z / (float)margin;
  if (iz < nz - 1 && z == 0 && mz > 0) w = (float)(mz - 1) / (float)margin;
  if (iy > 0 && y < margin) w = (float)y / (float)margin;
  if (iy < ny - 1 && y == 0) w = (float)(margin - 1) / (float)margin;
  if (ix > 0 && x < margin) w = (float)x / (float)margin;
  if (ix < nx - 1 && x == 0) w = (float)(margin - 1) / (float)margin;
  return w;
}

__global__ void __launch_bounds__(256) stitch_ramp_kernel(StitchRampArgs a) {
  // 4 consecutive x voxels per thread (one 16-byte load per covering patch when the run is inside the patch row and
  // aligned); per voxel the accumulation order is the reference's patch order z -> y -> x
  const int W4 = (a.W + 3) / 4;
  const long long total = (long long)a.V * a.C * a.Z * a.H * W4;
  const long long pvol = (long long)a.pd * a.ph * a.pw;
  const int npv = a.nz * a.ny * a.nx;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int x4 = (int)(r % W4) * 4; r /= W4;
    const int y = (int)(r % a.H); r /= a.H;
    const int z = (int)(r % a.Z); r /= a.Z;
    const int c = (int)(r % a.C); r /= a.C;
    const int v = (int)r;
    float acc[4] = {0.f, 0.f, 0.f, 0.f}, wsum[4] = {0.f, 0.f, 0.f, 0.f};
    for (int i = 0; i < a.nz; ++i) {
      const int tz = z - a.zs[i];
      if (tz < 0 || tz >= a.pd) continue;
      for (int j = 0; j < a.ny; ++j) {
        const int ty = y - a.ys[j];
        if (ty < 0 || ty >= a.ph) continue;
        for (int k = 0; k < a.nx; ++k) {
          const int tx0 = x4 - a.xs[k];
          if (tx0 <= -4 || tx0 >= a.pw) continue;
          const long long n = (long long)v * npv + (i * a.ny + j) * a.nx + k;
          const float* t = a.tiles + (n * a.C + c) * pvol + ((long long)tz * a.ph + ty) * a.pw;
          float pv[4];
          const bool whole = tx0 >= 0 && tx0 + 4 <= a.pw;
          if (whole && ((reinterpret_cast<uintptr_t>(t + tx0) & 15) == 0)) {
            *reinterpret_cast<float4*>(pv) = __ldg(reinterpret_cast<const float4*>(t + tx0));
          } else {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const int tx = tx0 + q;
              pv[q] = (tx >= 0 && tx < a.pw) ? __ldg(t + tx) : 0.f;
            }
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const int tx = tx0 + q;
            if (tx < 0 || tx >= a.pw) continue;
            const float w = ramp_weight(tz, ty, tx, i, j, k, a.nz, a.ny, a.nx, a.margin);
            acc[q] = __fadd_rn(acc[q], __fmul_rn(pv[q], w));
            wsum[q] = __fadd_rn(wsum[q], w);
          }
        }
      }
    }
    float o4[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) o4[q] = wsum[q] > 0.f ? __fdiv_rn(acc[q], wsum[q]) : 0.f;
    float* o = a.out + ((((long long)v * a.C + c) * a.Z + z) * a.H + y) * a.W + x4;
    if (x4 + 4 <= a.W && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
      *reinterpret_cast<float4*>(o) = *reinterpret_cast<float4*>(o4);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (x4 + q < a.W) o[q] = o4[q];
    }
  }
}
int launch_stitch_ramp(const StitchRampArgs& a, cudaStream_t stream) {
  const long long total = (long long)a.V * a.C * a.Z * a.H * ((a.W + 3) / 4);
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  stitch_ramp_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

}  // namespace biu

// ================================================================================================
// Multi-output 3D variants (multi_output_unet3d/predict.py:104-125, 127-174): float32 normalisation
// of an integer-valued stack and float32 patch gather.
// ================================================================================================
namespace biu {

// np.percentile on a float32 array with a python-float q: quantile, virtual index, gamma and the lerp are float32.
__device__ float percentile_from_hist_f32(const unsigned long long* cum_sh, const unsigned int* hist, long long n,
                                          float q) {
  const float quant = __fdiv_rn(q, 100.0f);
  const float vi = __fmul_rn((float)(n - 1), quant);
  long long prev = (long long)floorf(vi);
  long long next = prev + 1;
  float gamma;
  if (vi >= (float)(n - 1)) {
    prev = n - 1; next = n - 1;
    gamma = __fsub_rn(vi, -1.0f);
  } else if (vi < 0.0f) {
    prev = 0; next = 0;
    gamma = vi;
  } else {
    gamma = __fsub_rn(vi, (float)prev);
  }
  auto kth = [&](long long k) -> int {
    int g = 0;
    while (g < 255 && (long long)cum_sh[g] <= k) ++g;
    long long c = g == 0 ? 0 : (long long)cum_sh[g - 1];
    int b = g * 256;
    for (; b < g * 256 + 255; ++b) {
      c += hist[b];
      if (c > k) break;
    }
    return b;
  };
  const float a = (float)kth(prev);
  const float b = (float)kth(next);
  const float diff = __fsub_rn(b, a);
  float r = __fadd_rn(a, __fmul_rn(diff, gamma));
  if (gamma >= 0.5f) r = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, gamma)));
  return r;
}

// lut[f][v] = float32 of the float64 expression the reference evaluates for a voxel of value v:
//   mode 0 ('single'):      (clip(v, lo, hi) - min) / (ptp + 1e-8)         :108-112
//   mode 1 ('first'/'all'): (clip(v, lo, hi) - lo) / (hi - lo + 1e-8)      :114-120
//   mode 2 (multi_output_unet/predict.py:128-151, all three modes): x = clip(v, lo, hi); x = x - min(x); x / max(x),
//           entirely in float32 (float32 percentiles, float32 stack)
// np.clip of the float32 stack with np.float64 bounds promotes to float64 (NEP 50), the store back into the
// float32 stack rounds once.
__global__ void __launch_bounds__(256) norm_lut_f32_kernel(const unsigned int* __restrict__ hist_bounds,
                                                            const unsigned int* __restrict__ hist_range,
                                                            long long bounds_stride, long long range_stride,
                                                            double q_lo, double q_hi, int mode,
                                                            float* __restrict__ lut, double* __restrict__ params) {
  __shared__ unsigned long long cum[256];
  __shared__ double sp[4];
  __shared__ int s_vmin, s_vmax;
  const int f = blockIdx.x;
  const unsigned int* hb = hist_bounds + (long long)f * bounds_stride;
  const unsigned int* hr = hist_range + (long long)f * range_stride;
  {
    unsigned long long s = 0;
    for (int i = 0; i < 256; ++i) s += hb[threadIdx.x * 256 + i];
    cum[threadIdx.x] = s;
  }
  if (threadIdx.x == 0) { s_vmin = kHistBins; s_vmax = -1; }
  __syncthreads();
  {
    int lo_b = kHistBins, hi_b = -1;
    for (int i = 0; i < 256; ++i) {
      const int b = threadIdx.x * 256 + i;
      if (hr[b]) { if (b < lo_b) lo_b = b; if (b > hi_b) hi_b = b; }
    }
    if (hi_b >= 0) { atomicMin(&s_vmin, lo_b); atomicMax(&s_vmax, hi_b); }
  }
  if (threadIdx.x == 0)
    for (int g = 1; g < 256; ++g) cum[g] += cum[g - 1];
  __syncthreads();
  if (threadIdx.x == 0) {
    const long long n = (long long)cum[255];
    double lo, hi, sub, den;
    if (mode == 0 || mode == 2) {
      // 'single' (:108-112): np.percentile(float32 array, python float) runs entirely in float32 (the quantile is
      // divided by np.float32(100)), and so do the clip, min, ptp and the division.
      const float lo_f = percentile_from_hist_f32(cum, hb, n, (float)q_lo);
      const float hi_f = percentile_from_hist_f32(cum, hb, n, (float)q_hi);
      const float cmin = fminf(fmaxf((float)s_vmin, lo_f), hi_f);
      const float cmax = fminf(fmaxf((float)s_vmax, lo_f), hi_f);
      lo = lo_f; hi = hi_f; sub = cmin;
      den = mode == 0 ? __fadd_rn(__fsub_rn(cmax, cmin), 1e-8f) : __fsub_rn(cmax, cmin);
    } else {
      lo = percentile_from_hist(cum, hb, n, q_lo);
      hi = percentile_from_hist(cum, hb, n, q_hi);
      sub = lo;
      den = __dadd_rn(__dsub_rn(hi, lo), 1e-8);
    }
    sp[0] = lo; sp[1] = hi; sp[2] = sub; sp[3] = den;
    if (params) { params[f * 4 + 0] = lo; params[f * 4 + 1] = hi; params[f * 4 + 2] = sub; params[f * 4 + 3] = den; }
  }
  __syncthreads();
  const double lo = sp[0], hi = sp[1], sub = sp[2], den = sp[3];
  float* out = lut + (long long)f * kHistBins;
  for (int v = threadIdx.x; v < kHistBins; v += blockDim.x) {
    if (mode == 0 || mode == 2) {
      const float x = fminf(fmaxf((float)v, (float)lo), (float)hi);
      out[v] = __fdiv_rn(__fsub_rn(x, (float)sub), (float)den);
    } else {
      const double x = fmin(fmax((double)v, lo), hi);
      out[v] = __double2float_rn(__ddiv_rn(__dsub_rn(x, sub), den));
    }
  }
}

int launch_norm_lut_f32(const unsigned int* hist_bounds, const unsigned int* hist_range, long long bounds_stride,
                        long long range_stride, int frames, double q_lo, double q_hi, int mode, float* lut,
                        double* params, cudaStream_t stream) {
  norm_lut_f32_kernel<<<frames, 256, 0, stream>>>(hist_bounds, hist_range, bounds_stride, range_stride, q_lo, q_hi,
                                                  mode, lut, params);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

template <typename T>
__global__ void __launch_bounds__(256) apply_lut_f32_kernel(const T* __restrict__ img, long long n_per_frame,
                                                             const float* __restrict__ lut, long long lut_stride,
                                                             float* __restrict__ out, int blocks_per_frame) {
  const int frame = blockIdx.x / blocks_per_frame;
  const int blk = blockIdx.x % blocks_per_frame;
  const T* src = img + (long long)frame * n_per_frame;
  float* dst = out + (long long)frame * n_per_frame;
  const float* l = lut + (long long)frame * lut_stride;
  const long long stride = (long long)blocks_per_frame * blockDim.x;
  const long long n4 = (((uintptr_t)src & 7) == 0 && ((uintptr_t)dst & 15) == 0) ? n_per_frame / 4 : 0;
  for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < n4; i += stride) {
    T e[4];
    if (sizeof(T) == 2) *reinterpret_cast<uint2*>(e) = __ldg(reinterpret_cast<const uint2*>(src) + i);
    else *reinterpret_cast<uint32_t*>(e) = __ldg(reinterpret_cast<const uint32_t*>(src) + i);
    *reinterpret_cast<float4*>(dst + 4 * i) = make_float4(__ldg(l + e[0]), __ldg(l + e[1]), __ldg(l + e[2]), __ldg(l + e[3]));
  }
  for (long long i = n4 * 4 + (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame; i += stride)
    dst[i] = __ldg(l + src[i]);
}

int launch_apply_lut_f32(const void* img, int dtype_bytes, long long n_per_frame, int frames, const float* lut,
                         long long lut_stride, float* out, cudaStream_t stream) {
  BIU_REQUIRE(dtype_bytes == 1 || dtype_bytes == 2, "apply_lut_f32: only uint8/uint16 input");
  long long work = ceil_div_ll(n_per_frame, 256LL * 4 * 4);
  int bpf = (int)(work < 1 ? 1 : (work > 1184 ? 1184 : work));
  if (dtype_bytes == 2)
    apply_lut_f32_kernel<uint16_t><<<frames * bpf, 256, 0, stream>>>((const uint16_t*)img, n_per_frame, lut, lut_stride, out, bpf);
  else
    apply_lut_f32_kernel<uint8_t><<<frames * bpf, 256, 0, stream>>>((const uint8_t*)img, n_per_frame, lut, lut_stride, out, bpf);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// float32 patch gather, patches always inside the volume (patch = min(volume, max_patch), :129-131). Flips of `xform`
// (test-time augmentation) as in gather_tiles_kernel; a float4 run of a mirrored row is reversed in registers.
__global__ void __launch_bounds__(256) gather_tiles_f32_kernel(const float* __restrict__ src, int F, int Z, int H, int W,
                                                               const int* __restrict__ zs, const int* __restrict__ ys,
                                                               const int* __restrict__ xs, int nz, int ny, int nx, int pd,
                                                               int ph, int pw, float* __restrict__ dst, int xform) {
  // 4 consecutive x per thread (pw is a multiple of 4: patch extents are multiples of 8 / 16)
  const long long total = (long long)F * nz * ny * nx * pd * ph * pw;
  const bool fx = xform & XF_FLIP_X, fy = xform & XF_FLIP_Y, fz = xform & XF_FLIP_Z;
  for (long long idx = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4; idx < total;
       idx += (long long)gridDim.x * blockDim.x * 4) {
    long long r = idx;
    const int x = (int)(r % pw); r /= pw;
    const int y = (int)(r % ph); r /= ph;
    const int z = (int)(r % pd); r /= pd;
    const int ix = (int)(r % nx); r /= nx;
    const int iy = (int)(r % ny); r /= ny;
    const int iz = (int)(r % nz); r /= nz;
    const int f = (int)r;
    int zz = zs[iz] + (fz ? pd - 1 - z : z), yy = ys[iy] + (fy ? ph - 1 - y : y);
    if (zz >= Z) zz = reflect_index(zz, Z);      // np.pad(..., 'reflect') at the far end (multi_output_unet/predict.py:172),
    if (yy >= H) yy = reflect_index(yy, H);      // periodic like numpy's when the pad exceeds the extent
    const float* row = src + (((long long)f * Z + zz) * H + yy) * W;
    const int sx0 = xs[ix] + (fx ? pw - 4 - x : x);
    float v[4];
    if (sx0 + 4 <= W && ((reinterpret_cast<uintptr_t>(row + sx0) & 15) == 0)) {
      *reinterpret_cast<float4*>(v) = __ldg(reinterpret_cast<const float4*>(row + sx0));
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        int xx = sx0 + q;
        if (xx >= W) xx = reflect_index(xx, W);
        v[q] = __ldg(row + xx);
      }
    }
    if (fx) { float t0 = v[0], t1 = v[1]; v[0] = v[3]; v[1] = v[2]; v[2] = t1; v[3] = t0; }
    *reinterpret_cast<float4*>(dst + idx) = *reinterpret_cast<float4*>(v);
  }
}
int launch_gather_tiles_f32(const float* src, int F, int Z, int H, int W, const int* zs, const int* ys, const int* xs,
                            int nz, int ny, int nx, int pd, int ph, int pw, float* dst, cudaStream_t stream, int xform) {
  BIU_REQUIRE(pw % 4 == 0, "gather_tiles_f32: patch width must be a multiple of 4 (got %d)", pw);
  if (xform & XF_TRANSPOSE) {
    GatherArgs a{src, 4, nullptr, 0, F, Z, H, W, 0, zs, ys, xs, nz, ny, nx, pd, ph, pw, nullptr, xform};
    if (int rc = check_xform(a)) return rc;
    launch_gather_transposed<float, float>(a, dst, stream);
    BIU_CHECK_CUDA(cudaGetLastError());
    count_launch();
    return 0;
  }
  BIU_REQUIRE(xform >= 0 && xform <= (XF_FLIP_X | XF_FLIP_Y | XF_FLIP_Z), "gather_tiles_f32: bad transform %d", xform);
  const long long total = (long long)F * nz * ny * nx * pd * ph * pw / 4;
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  gather_tiles_f32_kernel<<<(int)blocks, 256, 0, stream>>>(src, F, Z, H, W, zs, ys, xs, nz, ny, nx, pd, ph, pw, dst,
                                                           xform);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// multi_output_unet/predict.py:230-285: margin-weighted mean of the float16 result patches. A patch has weight 1
// except on its first / last `margin` rows and columns where a neighbouring patch exists (weight 0); pixels no
// patch covers with weight > 0 get `*fill` (the global mean of the result patches). Patches are taken through the
// table src_index[(image, j, k)] because the reference indexes its flat patch list as image*N_per_img + j*N_y + k
// whatever the sliding-window count was. Accumulation in (j, k) order, float32, as numpy does.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) stitch_margin_kernel(StitchMarginArgs a) {
  const long long total = (long long)a.T * a.C * a.H * a.W;
  const float fill = __ldg(a.fill);
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int x = (int)(r % a.W); r /= a.W;
    const int y = (int)(r % a.H); r /= a.H;
    const int c = (int)(r % a.C); r /= a.C;
    const int i = (int)r;
    float acc = 0.f, wsum = 0.f;
    for (int j = 0; j < a.ny; ++j) {
      const int dy = y - a.ys[j];
      if (dy < 0 || dy >= a.ph) continue;
      const bool wy = !((j > 0 && dy < a.margin) || (j < a.ny - 1 && dy >= a.ph - a.margin));
      for (int k = 0; k < a.nx; ++k) {
        const int dx = x - a.xs[k];
        if (dx < 0 || dx >= a.pw) continue;
        const bool wx = !((k > 0 && dx < a.margin) || (k < a.nx - 1 && dx >= a.pw - a.margin));
        const float w = (wy && wx) ? 1.f : 0.f;
        const long long p = a.src_index[((long long)i * a.ny + j) * a.nx + k];
        const float v = __half2float(__float2half_rn(__ldg(a.tiles + ((p * a.C + c) * a.ph + dy) * a.pw + dx)));
        acc = __fadd_rn(acc, __fmul_rn(v, w));
        wsum += w;
      }
    }
    a.out[idx] = wsum > 0.f ? __fdiv_rn(acc, wsum) : fill;
  }
}
int launch_stitch_margin(const StitchMarginArgs& a, cudaStream_t stream) {
  const long long total = (long long)a.T * a.C * a.H * a.W;
  long long blocks = ceil_div_ll(total, 256);
  if (blocks > 148LL * 32) blocks = 148LL * 32;
  if (blocks < 1) blocks = 1;
  stitch_margin_kernel<<<(int)blocks, 256, 0, stream>>>(a);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// float32 stacks (unet/predict.py:122-150 on a float image: percentiles, clip, -min, /max*255 all in float32).
// Exact order statistics by a two-level radix select on the order-preserving 32-bit key of the float:
//   fkey_hi16 -> uint16 image of the keys' upper halves, histogrammed by histogram_kernel (shared with the integer
//   path, incl. hist_sum for stack-wide statistics); fkey_select picks, per statistics set, the upper-half bins that
//   hold the six ranks needed (two neighbours for each percentile, minimum, maximum); fkey_hist_lo histograms the
//   lower halves of the elements in those bins; fkey_params resolves the six floats and evaluates numpy's float32
//   percentile lerp; normalize_f32_kernel applies the reference's expression element-wise.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t fkey(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float fkey_inv(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__global__ void __launch_bounds__(256) fkey_hi16_kernel(const float* __restrict__ img, long long n, uint16_t* __restrict__ hi) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    hi[i] = (uint16_t)(fkey(__ldg(img + i)) >> 16);
}

struct FkeySel {              // per statistics set
  int bin[6];                 // upper-half bin of: lo.prev, lo.next, hi.prev, hi.next, min, max
  long long res[6];           // rank inside that bin
  float gamma[2];
};

// rank -> (bin, rank within bin) over a 65536-bin histogram with 256 group sums in shared memory
__device__ void fkey_rank_to_bin(const unsigned long long* cum_sh, const unsigned int* hist, long long k, int* bin, long long* res) {
  int g = 0;
  while (g < 255 && (long long)cum_sh[g] <= k) ++g;
  long long c = g == 0 ? 0 : (long long)cum_sh[g - 1];
  int b = g * 256;
  for (; b < g * 256 + 255; ++b) {
    if (c + hist[b] > k) break;
    c += hist[b];
  }
  *bin = b; *res = k - c;
}

__global__ void __launch_bounds__(256) fkey_select_kernel(const unsigned int* __restrict__ hist_bounds,
                                                          const unsigned int* __restrict__ hist_range,
                                                          long long bounds_stride, long long range_stride, float q_lo,
                                                          float q_hi, FkeySel* __restrict__ sel) {
  __shared__ unsigned long long cum_b[256], cum_r[256];
  const int s = blockIdx.x;
  const unsigned int* hb = hist_bounds + (long long)s * bounds_stride;
  const unsigned int* hr = hist_range + (long long)s * range_stride;
  unsigned long long sb = 0, sr = 0;
  for (int i = 0; i < 256; ++i) { sb += hb[threadIdx.x * 256 + i]; sr += hr[threadIdx.x * 256 + i]; }
  cum_b[threadIdx.x] = sb; cum_r[threadIdx.x] = sr;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int g = 1; g < 256; ++g) { cum_b[g] += cum_b[g - 1]; cum_r[g] += cum_r[g - 1]; }
    const long long nb = (long long)cum_b[255], nr = (long long)cum_r[255];
    FkeySel o;
    const float qs[2] = {q_lo, q_hi};
    for (int w = 0; w < 2; ++w) {        // np.percentile(float32 array, python float): float32 index arithmetic
      const float vi = __fmul_rn((float)(nb - 1), __fdiv_rn(qs[w], 100.0f));
      long long prev = (long long)floorf(vi), next = prev + 1;
      float gamma;
      if (vi >= (float)(nb - 1)) { prev = nb - 1; next = nb - 1; gamma = __fsub_rn(vi, -1.0f); }
      else if (vi < 0.0f) { prev = 0; next = 0; gamma = vi; }
      else gamma = __fsub_rn(vi, (float)prev);
      if (next > nb - 1) next = nb - 1;
      fkey_rank_to_bin(cum_b, hb, prev, &o.bin[2 * w], &o.res[2 * w]);
      fkey_rank_to_bin(cum_b, hb, next, &o.bin[2 * w + 1], &o.res[2 * w + 1]);
      o.gamma[w] = gamma;
    }
    fkey_rank_to_bin(cum_r, hr, 0, &o.bin[4], &o.res[4]);
    fkey_rank_to_bin(cum_r, hr, nr - 1, &o.bin[5], &o.res[5]);
    sel[s] = o;
  }
}

// hist_lo[set][6][65536]: lower key halves of the elements whose upper half is one of the set's six bins. A frame
// contributes to the percentile ranks (0..3) of its set only if frame < bounds_frames or the sets are per frame.
__global__ void __launch_bounds__(256) fkey_hist_lo_kernel(const float* __restrict__ img, long long n_per_frame,
                                                           int frames, const FkeySel* __restrict__ sel, int per_frame,
                                                           int bounds_frames, unsigned int* __restrict__ hist_lo,
                                                           int blocks_per_frame) {
  const int frame = blockIdx.x / blocks_per_frame, blk = blockIdx.x % blocks_per_frame;
  const int set = per_frame ? frame : 0;
  const FkeySel sl = sel[set];
  const bool bounds_ok = per_frame || frame < bounds_frames;
  unsigned int* h = hist_lo + (long long)set * 6 * kHistBins;
  const float* src = img + (long long)frame * n_per_frame;
  for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame; i += (long long)blocks_per_frame * blockDim.x) {
    const uint32_t k = fkey(__ldg(src + i));
    const int hi = (int)(k >> 16);
#pragma unroll
    for (int r = 0; r < 6; ++r)
      if (hi == sl.bin[r] && (r >= 4 || bounds_ok)) atomicAdd(&h[(long long)r * kHistBins + (k & 0xffffu)], 1u);
  }
}

// params[set] = {lo, hi, mn, mx} (float32): lo / hi = percentiles, mn = min(clip(img)), mx = max(clip(img) - mn)
__global__ void __launch_bounds__(192) fkey_params_kernel(const FkeySel* __restrict__ sel, const unsigned int* __restrict__ hist_lo,
                                                          float* __restrict__ params) {
  __shared__ float vals[6];
  const int s = blockIdx.x;
  const FkeySel sl = sel[s];
  if (threadIdx.x < 6) {
    const int r = threadIdx.x;
    const unsigned int* h = hist_lo + ((long long)s * 6 + r) * kHistBins;
    long long c = 0;
    int b = 0;
    for (; b < kHistBins - 1; ++b) {
      if (c + h[b] > sl.res[r]) break;
      c += h[b];
    }
    vals[r] = fkey_inv(((uint32_t)sl.bin[r] << 16) | (uint32_t)b);
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float pr[2];
    for (int w = 0; w < 2; ++w) {
      const float a = vals[2 * w], b = vals[2 * w + 1], g = sl.gamma[w];
      const float diff = __fsub_rn(b, a);
      float r = __fadd_rn(a, __fmul_rn(diff, g));
      if (g >= 0.5f) r = __fsub_rn(b, __fmul_rn(diff, __fsub_rn(1.0f, g)));
      pr[w] = r;
    }
    const float cmin = fminf(fmaxf(vals[4], pr[0]), pr[1]);
    const float cmax = fminf(fmaxf(vals[5], pr[0]), pr[1]);
    params[s * 4 + 0] = pr[0]; params[s * 4 + 1] = pr[1]; params[s * 4 + 2] = cmin; params[s * 4 + 3] = __fsub_rn(cmax, cmin);
  }
}

// out = uint8(trunc(float32(((clip(x, lo, hi) - mn) / mx) * 255 [255 - .]))), optionally also the float32 value
__global__ void __launch_bounds__(256) normalize_f32_kernel(const float* __restrict__ img, long long n_per_frame, int frames,
                                                            const float* __restrict__ params, int per_frame, int invert,
                                                            uint8_t* __restrict__ out_u8, float* __restrict__ out_f32,
                                                            int blocks_per_frame) {
  const int frame = blockIdx.x / blocks_per_frame, blk = blockIdx.x % blocks_per_frame;
  const float* pp = params + (per_frame ? frame : 0) * 4;
  const float lo = pp[0], hi = pp[1], mn = pp[2], mx = pp[3];
  const long long base = (long long)frame * n_per_frame;
  for (long long i = (long long)blk * blockDim.x + threadIdx.x; i < n_per_frame; i += (long long)blocks_per_frame * blockDim.x) {
    float x = fminf(fmaxf(__ldg(img + base + i), lo), hi);
    x = __fsub_rn(x, mn);
    x = __fmul_rn(__fdiv_rn(x, mx), 255.0f);
    if (invert) x = __fsub_rn(255.0f, x);
    if (out_f32) out_f32[base + i] = x;
    out_u8[base + i] = (uint8_t)(int)x;
  }
}

int launch_normalize_f32(const NormF32Args& a, cudaStream_t stream) {
  BIU_REQUIRE(a.mode >= 0 && a.mode <= 2, "normalize_f32: mode must be 0 (single), 1 (first) or 2 (all)");
  const long long n = a.n_per_frame * a.frames;
  const int per_frame = a.mode == 0 ? 1 : 0;
  const int sets = per_frame ? a.frames : 1;
  uint16_t* hi16 = reinterpret_cast<uint16_t*>(a.scratch);                                   // [n]
  unsigned int* hist = reinterpret_cast<unsigned int*>(a.scratch + ((n * 2 + 255) & ~255LL)); // [frames][65536]
  unsigned int* hist_tot = hist + (long long)a.frames * kHistBins;                           // [65536]
  unsigned int* hist_lo = hist_tot + kHistBins;                                              // [sets][6][65536]
  FkeySel* sel = reinterpret_cast<FkeySel*>(hist_lo + (long long)sets * 6 * kHistBins);      // [sets]
  long long blocks = ceil_div_ll(n, 256 * 8);
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (blocks < 1) blocks = 1;
  fkey_hi16_kernel<<<(int)blocks, 256, 0, stream>>>(a.img, n, hi16);
  BIU_CHECK_CUDA(cudaMemsetAsync(hist, 0, ((long long)(a.frames + 1 + sets * 6) * kHistBins) * sizeof(unsigned int), stream));
  if (int rc = launch_histogram(hi16, 2, a.n_per_frame, a.frames, hist, stream)) return rc;
  const unsigned int* hb = hist; const unsigned int* hr = hist;
  long long bs = kHistBins, rs = kHistBins;
  if (!per_frame) {
    if (int rc = launch_hist_sum(hist, a.frames, hist_tot, stream)) return rc;
    hr = hist_tot; rs = 0;
    hb = a.mode == 2 ? hist_tot : hist; bs = 0;          // 'first': bounds from frame 0 only
  }
  fkey_select_kernel<<<sets, 256, 0, stream>>>(hb, hr, bs, rs, (float)a.q_lo, (float)a.q_hi, sel);
  long long bpf = ceil_div_ll(a.n_per_frame, 256 * 16);
  if (bpf > 296) bpf = 296;
  if (bpf < 1) bpf = 1;
  fkey_hist_lo_kernel<<<(int)(a.frames * bpf), 256, 0, stream>>>(a.img, a.n_per_frame, a.frames, sel, per_frame,
                                                                 a.mode == 1 ? 1 : a.frames, hist_lo, (int)bpf);
  fkey_params_kernel<<<sets, 192, 0, stream>>>(sel, hist_lo, a.params);
  normalize_f32_kernel<<<(int)(a.frames * bpf), 256, 0, stream>>>(a.img, a.n_per_frame, a.frames, a.params, per_frame,
                                                                  a.invert, a.out_u8, a.out_f32, (int)bpf);
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch(5);
  return 0;
}

long long normalize_f32_scratch_bytes(long long n_per_frame, int frames) {
  const long long n = n_per_frame * frames;
  return ((n * 2 + 255) & ~255LL) + ((long long)(frames + 1 + frames * 6) * kHistBins) * 4 + (long long)frames * sizeof(FkeySel) + 256;
}

}  // namespace biu
