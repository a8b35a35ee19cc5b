// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a).
//
// One CTA computes a 128-pixel x n_blk-channel output tile:
//   D[128 pixels, n_blk] = sum over (channel chunk, filter tap) A[128, ck] * B[n_blk, ck]^T
// * A: a TMA box (ck channels, bw, bh, bd, bb pixels; bw*bh*bd*bb = 128) of the NHWC/NDHWC activation tensor,
//      shifted by the tap offset. Out-of-bounds coordinates are zero-filled by TMA, which is exactly the
//      convolution's zero padding; every image tile is its own index on the outermost dim, so nothing leaks
//      between tiles (reference: each tile is an independent forward, unet/predict.py:191-201).
// * B: a TMA box (ck, n_blk, 1) of the packed weights [tap][Cout][Cin].
// * accumulator: fp32 in TMEM; epilogue = folded BatchNorm scale/shift + LeakyReLU (unet/unet.py:54-60),
//      or bias + 2x pixel-shuffle for ConvTranspose(k=2,s=2) (unet/unet.py:38-47),
//      or the block followed by the 1x1 head + activation (unet/unet.py:50-52,104).
// Warp roles: warp 0 TMA producer, warp 1 TMEM allocator + MMA issuer, warps 2-5 epilogue.
#pragma once
#include "common.cuh"

namespace biu {

enum EpiMode { EPI_CONV = 0, EPI_UP = 1, EPI_HEAD = 2 };
enum HeadAct { ACT_NONE = 0, ACT_SIGMOID = 1, ACT_TANH = 2, ACT_RELU = 3 };

constexpr int kMaxHead = 8;
constexpr int kMaxStages = 8;

struct ConvTcParams {
  int W, H, D, B;                            // activation extents (output = input extents, stride 1)
  int lbw, lbh, lbd, lbb;                    // log2 of the pixel box; sums to 7
  int tiles_w, tiles_h, tiles_d, tiles_b;    // tile grid
  int kw, kh, kd;                            // filter extents (3 or 1)
  int cin_chunks, ck;                        // K chunks per tap, elements per chunk
  int row_bytes;                             // ck * element size: 32, 64 or 128 (== swizzle span)
  int n_blk;                                 // output channels per CTA (multiple of 16, <= 256)
  int stages;
  int mode;
  float slope;
  const float* scale;                        // [n_total]
  const float* shift;                        // [n_total]
  void* out;                                 // NHWC destination (bf16 / fp16 or fp32); may be null in EPI_HEAD
  int out_ctot, out_coff;
  int up_cout, up_dims;                      // EPI_UP
  int head_n;                                // EPI_HEAD
  const float* head_w;                       // [head_n][n_blk]
  const float* head_b;                       // [head_n]
  int head_act[kMaxHead];
  float* out_val;                            // planar [B][head_n][D][H][W] activated head output (optional)
  uint8_t* out_u8;                           // planar, trunc(val * 255) (optional)
};

__device__ __forceinline__ float apply_head_act(float v, int act) {
  switch (act) {
    case ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
    case ACT_TANH: return tanhf(v);
    case ACT_RELU: return fmaxf(v, 0.0f);
    default: return v;
  }
}

__device__ __forceinline__ float round_tf32(float v) {
  uint32_t u;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
  return __uint_as_float(u);
}

template <int FMT>
__global__ void __launch_bounds__(192) conv_tc_kernel(const __grid_constant__ CUtensorMap tmA,
                                                      const __grid_constant__ CUtensorMap tmB,
                                                      const ConvTcParams p) {
  constexpr int ESZ = fmt_esz(FMT);
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t full_bar[kMaxStages];
  __shared__ uint64_t empty_bar[kMaxStages];
  __shared__ uint64_t tmem_full_bar;
  __shared__ uint32_t tmem_slot;

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  // 1024-byte aligned operand ring (required by the 128B swizzle atom).
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t a_bytes = 128u * p.row_bytes;
  const uint32_t b_bytes = ((uint32_t)p.n_blk * p.row_bytes + 1023u) & ~1023u;
  const uint32_t stage_bytes = a_bytes + b_bytes;
  const uint32_t tx_bytes = 128u * p.row_bytes + (uint32_t)p.n_blk * p.row_bytes;

  // tile coordinates
  int t = blockIdx.x;
  const int tx = t % p.tiles_w; t /= p.tiles_w;
  const int ty = t % p.tiles_h; t /= p.tiles_h;
  const int tz = t % p.tiles_d; t /= p.tiles_d;
  const int tb = t;
  const int x0 = tx << p.lbw, y0 = ty << p.lbh, z0 = tz << p.lbd, b0 = tb << p.lbb;
  const int n0 = blockIdx.y * p.n_blk;

  const int taps = p.kw * p.kh * p.kd;
  const int num_kb = p.cin_chunks * taps;

  uint32_t ncols = 32;
  while (ncols < (uint32_t)p.n_blk) ncols <<= 1;

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&tmem_full_bar, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_slot, ncols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ===================================== TMA producer =====================================
    if (elect_one()) {
      int kb = 0;
      for (int ch = 0; ch < p.cin_chunks; ++ch) {
        int tap = 0;
        for (int dz = 0; dz < p.kd; ++dz)
          for (int dy = 0; dy < p.kh; ++dy)
            for (int dx = 0; dx < p.kw; ++dx, ++tap, ++kb) {
              const int s = kb % p.stages;
              const uint32_t ph = (kb / p.stages) & 1;
              mbar_wait(&empty_bar[s], ph ^ 1, 0x100 + s);
              mbar_arrive_expect_tx(&full_bar[s], tx_bytes);
              const uint32_t a_dst = smem_base + s * stage_bytes;
              const uint32_t b_dst = a_dst + a_bytes;
              asm volatile(
                  "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
                  "%4, %5, %6, %7}], [%2];" ::"r"(a_dst),
                  "l"(reinterpret_cast<uint64_t>(&tmA)), "r"(smem_u32(&full_bar[s])), "r"(ch * p.ck),
                  "r"(x0 + dx - (p.kw >> 1)), "r"(y0 + dy - (p.kh >> 1)), "r"(z0 + dz - (p.kd >> 1)), "r"(b0)
                  : "memory");
              asm volatile(
                  "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, "
                  "%4, %5}], [%2];" ::"r"(b_dst),
                  "l"(reinterpret_cast<uint64_t>(&tmB)), "r"(smem_u32(&full_bar[s])), "r"(ch * p.ck), "r"(n0),
                  "r"(tap)
                  : "memory");
            }
      }
    }
  } else if (warp == 1) {
    // ====================================== MMA issuer ======================================
    if (elect_one()) {
      const uint32_t layout = p.row_bytes == 128 ? 2u : (p.row_bytes == 64 ? 4u : 6u);
      const uint32_t sbo = 8u * p.row_bytes;
      const uint32_t idesc = make_idesc(fmt_idesc(FMT), (uint32_t)p.n_blk);
      const int ksteps = p.row_bytes / 32;
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % p.stages;
        const uint32_t ph = (kb / p.stages) & 1;
        mbar_wait(&full_bar[s], ph, 0x200 + s);
        tc_fence_after();
        const uint32_t a_addr = smem_base + s * stage_bytes;
        const uint32_t b_addr = a_addr + a_bytes;
        for (int k = 0; k < ksteps; ++k) {
          const uint64_t adesc = make_smem_desc(a_addr + k * 32, sbo, layout);
          const uint64_t bdesc = make_smem_desc(b_addr + k * 32, sbo, layout);
          if (ESZ == 2)
            tc_mma_f16(tmem_base, adesc, bdesc, idesc, (kb | k) != 0);
          else
            tc_mma_tf32(tmem_base, adesc, bdesc, idesc, (kb | k) != 0);
        }
        tc_commit(&empty_bar[s]);  // frees the smem slot once these MMAs have read it
      }
      tc_commit(&tmem_full_bar);   // accumulator complete
    }
  } else {
    // ======================================= epilogue =======================================
    mbar_wait(&tmem_full_bar, 0, 0x300);
    tc_fence_after();
    const int grp = warp & 3;                   // TMEM lane quarter this warp may read
    const int m = grp * 32 + lane;              // accumulator row = pixel within the box
    int r = m;
    const int px = x0 + (r & ((1 << p.lbw) - 1)); r >>= p.lbw;
    const int py = y0 + (r & ((1 << p.lbh) - 1)); r >>= p.lbh;
    const int pz = z0 + (r & ((1 << p.lbd) - 1)); r >>= p.lbd;
    const int pb = b0 + r;
    const bool valid = px < p.W && py < p.H && pz < p.D && pb < p.B;
    const uint32_t trow = tmem_base + ((uint32_t)(grp * 32) << 16);

    float hacc[kMaxHead];
#pragma unroll
    for (int h = 0; h < kMaxHead; ++h) hacc[h] = 0.f;

    const long long pix = (((long long)pb * p.D + pz) * p.H + py) * p.W + px;

    for (int c0 = 0; c0 < p.n_blk; c0 += 16) {
      uint32_t acc[16];
      tmem_ld16(trow + c0, acc);
      tmem_ld_wait();
      float v[16];
      const int n = n0 + c0;
      if (p.mode == EPI_UP) {
#pragma unroll
        for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(acc[i]) + __ldg(p.shift + n + i);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float a = fmaf(__uint_as_float(acc[i]), __ldg(p.scale + n + i), __ldg(p.shift + n + i));
          v[i] = a > 0.f ? a : a * p.slope;
        }
      }
      if (p.mode == EPI_HEAD) {
        for (int h = 0; h < p.head_n; ++h) {
          float s = hacc[h];
#pragma unroll
          for (int i = 0; i < 16; ++i) s = fmaf(v[i], __ldg(p.head_w + h * p.n_blk + c0 + i), s);
          hacc[h] = s;
        }
      }
      if (valid && p.out != nullptr) {
        long long off;
        if (p.mode == EPI_UP) {
          const int q = n / p.up_cout, co = n - q * p.up_cout;
          const int ax = q & 1, ay = (q >> 1) & 1, az = (p.up_dims == 3) ? (q >> 2) & 1 : 0;
          const int oW = 2 * p.W, oH = 2 * p.H, oD = (p.up_dims == 3) ? 2 * p.D : p.D;
          const int oz = (p.up_dims == 3) ? 2 * pz + az : pz;
          const long long opix = (((long long)pb * oD + oz) * oH + (2 * py + ay)) * oW + (2 * px + ax);
          off = opix * p.out_ctot + p.out_coff + co;
        } else {
          off = pix * p.out_ctot + p.out_coff + n;
        }
        if (ESZ == 2) {
          uint32_t w[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) w[i] = pack_half2<FMT>(v[2 * i], v[2 * i + 1]);
          uint4* dst = reinterpret_cast<uint4*>(reinterpret_cast<uint16_t*>(p.out) + off);
          dst[0] = make_uint4(w[0], w[1], w[2], w[3]);
          dst[1] = make_uint4(w[4], w[5], w[6], w[7]);
        } else {
          float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + off);
#pragma unroll
          for (int i = 0; i < 4; ++i)
            dst[i] = make_float4(round_tf32(v[4 * i]), round_tf32(v[4 * i + 1]), round_tf32(v[4 * i + 2]),
                                 round_tf32(v[4 * i + 3]));
        }
      }
    }
    if (p.mode == EPI_HEAD && valid) {
      const long long plane = (long long)p.D * p.H * p.W;
      const long long sp = ((long long)pz * p.H + py) * p.W + px;
      for (int h = 0; h < p.head_n; ++h) {
        const float val = apply_head_act(hacc[h] + __ldg(p.head_b + h), p.head_act[h]);
        const long long o = ((long long)pb * p.head_n + h) * plane + sp;
        if (p.out_val) p.out_val[o] = val;
        if (p.out_u8) p.out_u8[o] = (uint8_t)(val * 255.0f);  // unet/predict.py:200 truncating cast
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, ncols);
}

}  // namespace biu
