// Implicit-GEMM convolution on tcgen05 with a shared-memory HALO tile — persistent, warp-specialised.
//
// Work item ("tile") = a macro tile of 16 rows x (8*mt) columns of one image plane (mt MMA tiles of 16x8 = 128
// pixels) x n_blk output channels. A CTA (one per SM) walks tiles blockIdx.x, +gridDim.x, ...
// 3x3(x3) blocks (halo = 1): per input-channel chunk the A producer TMA-loads ONE halo tile (ck channels x
// (8*mt+2) x 18 x kd pixels; out of bounds = zero = the convolution's padding) and all 9 / 27 filter taps run out
// of it: the A operand of tap (dz,dy,dx), MMA tile j is the same shared-memory tile addressed at row
//     ((dz*18 + dy) * (8*mt+2) + 8*j + dx)
// with 8-row core-matrix groups (8*mt+2) rows apart (stride-byte-offset of the smem descriptor). The 128B / 64B /
// 32B TMA swizzle is a function of the absolute shared-memory address, so row-shifted starts need no re-layout
// (verified on B200 by tools/tc_probe.cu -> profiles/r01_tc_descriptor_probe.txt).
// Transposed convolutions k=2,s=2 (halo = 0): a plain GEMM with N = 2^dims * Cout over the same tile walk (one
// "tap", 16 x 8*mt pixel tile) and a pixel-shuffle store.
// Pipelines: halo ring (a_full/a_empty), weight-tile ring (b_full/b_empty), two TMEM accumulator stages
// (acc_full/acc_empty) so the epilogue of tile i overlaps the MMAs of tile i+1.
// Warp roles: 0 = halo (A) producer, 1 = TMEM alloc + MMA issuer, 2 = weight (B) producer, 4..11 = epilogue (two
// groups of four warps; a warp reads the TMEM lane quarter warp % 4).
// The MMA warp runs its loops warp-uniformly (descriptor arithmetic stays in uniform registers; only the
// tcgen05.mma / commit instructions are predicated on the elected lane): the single-thread form spent ~70 cycles
// of R2UR / address arithmetic per MMA, which bounded every layer with N <= 128 (tools/conv_bench.cu).
// Epilogue: per-channel scale/shift staged once per CTA in shared memory, TMEM loads software-pipelined against
// the math + stores of the previous chunk, optional fused 2x2 max-pool (warp shuffles) of the stored values.
#pragma once
#include "conv_tc.cuh"

namespace biu {

constexpr int kMaxBStages = 36;
constexpr int kMaxABufs = 3;
constexpr int kHaloThreads = 384;   // warps: 0 A producer, 1 MMA, 2 B producer, 3 idle, 4..11 epilogue

struct ConvHaloParams {
  int W, H, D, B;
  int mt;                          // MMA tiles (16x8 pixels) per work item along x
  int tiles_x, tiles_y;            // macro tiles per image plane
  int n_blocks;                    // output-channel blocks
  int nblk_inner;                  // work-item order: the output-channel block is the FASTEST index (see halo_decode)
  int total_tiles;                 // tiles_x * tiles_y * D * B * n_blocks
  int kd;                          // z taps: 1 (2D) or 3
  int halo;                        // 1: 3x3(x3) convolution, 0: single tap (transposed convolution as GEMM)
  int cin_chunks, ck, row_bytes;
  int n_blk, n_total;
  int a_bufs, b_stages;
  int b_resident;                  // all (chunk, tap) weight tiles of the single n-block fit the ring: loaded once
  int cta2;                        // CTA pairs: tiles t, t+1 of a pair share one tcgen05.mma.cta_group::2 of M = 256; every
                                   // CTA stages only n_blk / 2 rows of each weight tile (b_stage_bytes counts those)
  int stage_bytes;                 // shared memory reserved for the epilogue's transposed-store tiles (0 or 16 KB)
  uint32_t a_buf_bytes, b_stage_bytes;
  int mode;
  float slope;
  const float* scale;
  const float* shift;
  void* out;
  int out_ctot, out_coff;
  int up_cout, up_dims;            // EPI_UP
  void* pool_out;                  // EPI_CONV, 2D: fused MaxPool2d(2) of the stored activations (may be null)
  int pool_ctot, pool_coff;
  int head_n;
  const float* head_w;
  const float* head_b;
  int head_act[kMaxHead];
  float* out_val;
  uint8_t* out_u8;
  int dbg;                         // tools/conv_bench.cu only (BIU_DBG_KNOBS): 1 no stores, 2 no MMA, 4 no A loads,
                                   // 8 no epilogue, 16 no B loads
};

#ifdef BIU_DBG_KNOBS
#define BIU_DBG(p, bit) (((p).dbg & (bit)) != 0)
// cycle accounting of CTA 0 (tools/conv_bench.cu): slot += clock64() spent in a region
static __device__ unsigned long long g_halo_prof[32];
#define PROF_DECL(cond) long long _pt = 0; const bool _pon = blockIdx.x == 0 && (cond) && (p.dbg & 256)
#define PROF_T0() do { if (_pon) _pt = clock64(); } while (0)
#define PROF_ADD(slot) do { if (_pon) { long long _n = clock64(); g_halo_prof[slot] += (unsigned long long)(_n - _pt); _pt = _n; } } while (0)
#else
#define BIU_DBG(p, bit) false
#define PROF_DECL(cond)
#define PROF_T0()
#define PROF_ADD(slot)
#endif

struct HaloTile { int x0, y0, z0, b0, n0; };

__device__ __forceinline__ HaloTile halo_decode(const ConvHaloParams& p, int t) {
  HaloTile r;
  // Blocks whose weights stay resident walk all tiles of one output-channel block first. Where the weights are streamed
  // anyway (transposed convolutions with N = 4 * Cout in several blocks) the block index is the fastest one instead:
  // neighbouring CTAs work on the SAME pixels at the same time, so the input tile comes from DRAM once and from L2 for
  // the other blocks (up1 of Unet(32): 0.84 -> 0.2 GB read per 200 tiles).
  int nb = 0;
  if (p.nblk_inner) { nb = t % p.n_blocks; t /= p.n_blocks; }
  const int tx = t % p.tiles_x; t /= p.tiles_x;
  const int ty = t % p.tiles_y; t /= p.tiles_y;
  r.z0 = t % p.D; t /= p.D;
  r.b0 = t % p.B; t /= p.B;
  r.n0 = (p.nblk_inner ? nb : t) * p.n_blk;
  r.x0 = tx * 8 * p.mt;
  r.y0 = ty * 16;
  return r;
}

// tcgen05.mma with a compile-time accumulate flag (no predicate register to materialise per instruction)
template <int FMT, int ACC, bool CTA2 = false>
__device__ __forceinline__ void tc_mma_imm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  constexpr int ESZ = fmt_esz(FMT);               // 2: kind::f16 (bf16 and fp16 operands), 4: kind::tf32
  if (CTA2) {                           // one MMA of M = 256 over the CTA pair (issued by the leader CTA only)
    if (ESZ == 2) {
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "setp.ne.b32 p, %4, 0;\n"
          "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
          "}\n" ::"r"(tmem_d),
          "l"(adesc), "l"(bdesc), "r"(idesc), "n"(ACC)
          : "memory");
    } else {
      asm volatile(
          "{\n"
          ".reg .pred p;\n"
          "setp.ne.b32 p, %4, 0;\n"
          "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n"
          "}\n" ::"r"(tmem_d),
          "l"(adesc), "l"(bdesc), "r"(idesc), "n"(ACC)
          : "memory");
    }
  } else if (ESZ == 2) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "n"(ACC)
        : "memory");
  } else {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "n"(ACC)
        : "memory");
  }
}

// predicated single-lane issue from warp-uniform code
template <int FMT>
__device__ __forceinline__ void tc_mma_pred(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate, uint32_t issue) {
  constexpr int ESZ = fmt_esz(FMT);
  if (ESZ == 2) {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(issue)
        : "memory");
  } else {
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "setp.ne.b32 q, %5, 0;\n"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(issue)
        : "memory");
  }
}
__device__ __forceinline__ void tc_commit_pred(uint64_t* bar, uint32_t issue) {
  asm volatile(
      "{\n"
      ".reg .pred q;\n"
      "setp.ne.b32 q, %1, 0;\n"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(issue)
      : "memory");
}

// TMEM -> registers, CW (16 or 32) consecutive fp32 columns of this warp's lane quarter; completion is only
// guaranteed after tmem_wait_regs on the same array.
template <int CW>
__device__ __forceinline__ void tmem_ld_cw(uint32_t taddr, uint32_t (&r)[32]) {
  if (CW == 32) {
    tmem_ld32(taddr, r);
  } else {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  }
}
// tcgen05.wait::ld with the destination registers as in/out operands: nothing that reads them can be scheduled
// above the wait.
template <int CW>
__device__ __forceinline__ void tmem_wait_regs(uint32_t (&r)[32]) {
  if (CW == 32) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                   "+r"(r[15]), "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]),
                   "+r"(r[22]), "+r"(r[23]), "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]),
                   "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :
                 : "memory");
  } else {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]),
                   "+r"(r[15])
                 :
                 : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Epilogue (warps 4..11). Specialised at compile time on the mode so that one chunk is straight-line code:
//   MODE EPI_CONV: scale/shift + LeakyReLU -> NHWC store [+ POOL: fused MaxPool2d(2) of the stored values]
//   MODE EPI_UP  : bias -> pixel-shuffle store of the transposed convolution
//   MODE EPI_HEAD: block activation kept in registers, 1x1 head + activation -> planar float / uint8
// Work units = (MMA tile j, chunk of CW accumulator columns); the two warp groups take alternate units. With the
// fused head a thread needs the whole channel row of its pixel, so there the groups alternate MMA tiles instead.
// ---------------------------------------------------------------------------------------------------------------
template <int FMT>
__device__ __forceinline__ void epi_store16(char* dst, const float (&v)[16], uint32_t (&w)[8]) {
  if (fmt_esz(FMT) == 2) {
#pragma unroll
    for (int i = 0; i < 8; ++i) w[i] = pack_half2<FMT>(v[2 * i], v[2 * i + 1]);
    if (dst != nullptr) {
      uint4* d4 = reinterpret_cast<uint4*>(dst);
      d4[0] = make_uint4(w[0], w[1], w[2], w[3]);
      d4[1] = make_uint4(w[4], w[5], w[6], w[7]);
    }
  } else {
    if (dst != nullptr) {
      float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll
      for (int i = 0; i < 4; ++i) d4[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
    }
  }
}

template <int FMT, int CW, int MODE, bool POOL>
__device__ __forceinline__ void halo_epi_chunk(const ConvHaloParams& p, const uint32_t (&acc)[32], const float* s_sc,
                                               const float* s_sh, const float* s_hw, char* out_px, char* pool_px,
                                               int n, float (&hacc)[kMaxHead], int up_plane_elems, int up_row_elems,
                                               uint32_t stage, char* tr_ptr, long long tr_row_bytes, int tr_px_bytes,
                                               uint32_t tr_mask, int lane) {
  constexpr int ESZ = fmt_esz(FMT);
  // s_sc / s_sh / s_hw already point at the first channel of this chunk; out_px at the thread's pixel (channel of
  // the chunk for CONV, channel 0 of the output pixel (2y, 2x) for UP); nullptr = masked pixel.
  // stage != 0 (CW = 32, one destination pixel per thread): the 64 / 128 bytes of every pixel go through a
  // per-warp shared-memory tile (16-byte chunks XOR-swizzled, conflict free both ways) and are written back
  // transposed, lane = (pixel, chunk): one warp store covers 8 (bf16) / 4 (fp32) pixels x 64 / 128 contiguous bytes =
  // full 32-byte sectors instead of 32 scattered 16-byte pieces. tr_ptr: destination of (row 0, pixel column
  // lane / LPP, chunk lane % LPP) of the warp's 4 x 8 pixel group; tr_mask: bit r set when the pixel written by
  // write-back instruction r is inside the image.
#pragma unroll
  for (int q = 0; q < CW / 16; ++q) {
    float v[16];
#pragma unroll
    for (int i4 = 0; i4 < 4; ++i4) {
      const float4 sh = reinterpret_cast<const float4*>(s_sh + q * 16)[i4];
      float a0, a1, a2, a3;
      if (MODE == EPI_UP) {                           // transposed convolution: bias only
        a0 = __uint_as_float(acc[q * 16 + 4 * i4 + 0]) + sh.x;
        a1 = __uint_as_float(acc[q * 16 + 4 * i4 + 1]) + sh.y;
        a2 = __uint_as_float(acc[q * 16 + 4 * i4 + 2]) + sh.z;
        a3 = __uint_as_float(acc[q * 16 + 4 * i4 + 3]) + sh.w;
      } else {
        const float4 sc = reinterpret_cast<const float4*>(s_sc + q * 16)[i4];
        a0 = fmaf(__uint_as_float(acc[q * 16 + 4 * i4 + 0]), sc.x, sh.x);
        a1 = fmaf(__uint_as_float(acc[q * 16 + 4 * i4 + 1]), sc.y, sh.y);
        a2 = fmaf(__uint_as_float(acc[q * 16 + 4 * i4 + 2]), sc.z, sh.z);
        a3 = fmaf(__uint_as_float(acc[q * 16 + 4 * i4 + 3]), sc.w, sh.w);
        a0 = fmaxf(a0, a0 * p.slope);                 // LeakyReLU for 0 <= slope <= 1 (1: identity, 0: ReLU)
        a1 = fmaxf(a1, a1 * p.slope);
        a2 = fmaxf(a2, a2 * p.slope);
        a3 = fmaxf(a3, a3 * p.slope);
      }
      if (ESZ == 4) { a0 = round_tf32(a0); a1 = round_tf32(a1); a2 = round_tf32(a2); a3 = round_tf32(a3); }
      v[4 * i4 + 0] = a0; v[4 * i4 + 1] = a1; v[4 * i4 + 2] = a2; v[4 * i4 + 3] = a3;
    }
    if (MODE == EPI_HEAD) {
#pragma unroll
      for (int h = 0; h < kMaxHead; ++h) {
        if (h >= p.head_n) break;                     // uniform exit: no predicated-off work for absent heads
        const float4* hw4 = reinterpret_cast<const float4*>(s_hw + h * p.n_blk + q * 16);
        float sacc = hacc[h];
#pragma unroll
        for (int i4 = 0; i4 < 4; ++i4) {
          const float4 w = hw4[i4];
          sacc = fmaf(v[4 * i4 + 0], w.x, sacc);
          sacc = fmaf(v[4 * i4 + 1], w.y, sacc);
          sacc = fmaf(v[4 * i4 + 2], w.z, sacc);
          sacc = fmaf(v[4 * i4 + 3], w.w, sacc);
        }
        hacc[h] = sacc;
      }
      if (p.out == nullptr) continue;
    }
    uint32_t w[8];
    if (CW == 32 && stage != 0) {
      if (ESZ == 2) {
#pragma unroll
        for (int i = 0; i < 8; ++i) w[i] = pack_half2<FMT>(v[2 * i], v[2 * i + 1]);
        const uint32_t sw = (uint32_t)(lane >> 1) & 3u, row = stage + (uint32_t)lane * 64u;
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + (((2u * q) ^ sw) << 4)), "r"(w[0]), "r"(w[1]),
                     "r"(w[2]), "r"(w[3]) : "memory");
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + (((2u * q + 1u) ^ sw) << 4)), "r"(w[4]),
                     "r"(w[5]), "r"(w[6]), "r"(w[7]) : "memory");
      } else {                                      // fp32 storage: 128 bytes per pixel, 8 chunks, XOR with lane & 7
        const uint32_t sw = (uint32_t)lane & 7u, row = stage + (uint32_t)lane * 128u;
#pragma unroll
        for (int i = 0; i < 4; ++i)
          asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(row + (((4u * q + i) ^ sw) << 4)),
                       "r"(__float_as_uint(v[4 * i])), "r"(__float_as_uint(v[4 * i + 1])),
                       "r"(__float_as_uint(v[4 * i + 2])), "r"(__float_as_uint(v[4 * i + 3])) : "memory");
      }
    } else if (MODE == EPI_UP) {
      // channel n+16q of the GEMM = (kernel position qd, output channel co); qd = (az, ay, ax) bits
      const int nn = n + q * 16;
      const int qd = nn / p.up_cout, co = nn - qd * p.up_cout;
      const int off = (qd >> 2) * up_plane_elems + ((qd >> 1) & 1) * up_row_elems + (qd & 1) * p.out_ctot + co;
      epi_store16<FMT>(out_px ? out_px + (long long)off * ESZ : nullptr, v, w);
    } else {
      epi_store16<FMT>(out_px ? out_px + q * 16 * ESZ : nullptr, v, w);
    }
    if (POOL) {                                       // MaxPool2d(2) of the stored (rounded) values: x pairs are
      if (ESZ == 2) {                                 // lanes ^1, y pairs lanes ^8 (pixel = (lane >> 3, lane & 7))
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint32_t mm = max_half2<FMT>(w[i], __shfl_xor_sync(0xffffffffu, w[i], 1));
          w[i] = max_half2<FMT>(mm, __shfl_xor_sync(0xffffffffu, mm, 8));
        }
        if (pool_px != nullptr) {
          uint4* d4 = reinterpret_cast<uint4*>(pool_px + q * 16 * ESZ);
          d4[0] = make_uint4(w[0], w[1], w[2], w[3]);
          d4[1] = make_uint4(w[4], w[5], w[6], w[7]);
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          v[i] = fmaxf(v[i], __shfl_xor_sync(0xffffffffu, v[i], 1));
          v[i] = fmaxf(v[i], __shfl_xor_sync(0xffffffffu, v[i], 8));
        }
        if (pool_px != nullptr) {
          float4* d4 = reinterpret_cast<float4*>(pool_px + q * 16 * ESZ);
#pragma unroll
          for (int i = 0; i < 4; ++i) d4[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        }
      }
    }
  }
  if (CW == 32 && stage != 0) {
    constexpr int LPP = 2 * ESZ;                      // lanes (16-byte chunks) per pixel: 4 (bf16) or 8 (fp32)
    __syncwarp();
#pragma unroll
    for (int r = 0; r < LPP; ++r) {
      const uint32_t pp = (uint32_t)(r * (32 / LPP) + lane / LPP);          // pixel (pp >> 3, pp & 7) of the group
      const uint32_t sw = ESZ == 2 ? ((pp >> 1) & 3u) : (pp & 7u);
      uint32_t d0, d1, d2, d3;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                   : "=r"(d0), "=r"(d1), "=r"(d2), "=r"(d3)
                   : "r"(stage + pp * (uint32_t)(LPP * 16) + ((((uint32_t)lane & (LPP - 1)) ^ sw) << 4))
                   : "memory");
      // bf16: instruction r = row r, column lane / 4; fp32: row r / 2, column (r & 1) * 4 + lane / 8
      char* dst = ESZ == 2 ? tr_ptr + r * tr_row_bytes : tr_ptr + (r >> 1) * tr_row_bytes + (r & 1) * 4 * tr_px_bytes;
      if (tr_ptr != nullptr && ((tr_mask >> r) & 1u)) *reinterpret_cast<uint4*>(dst) = make_uint4(d0, d1, d2, d3);
    }
    __syncwarp();
  }
}

template <int FMT, int CW, int MODE, bool POOL, bool CTA2>
__device__ __forceinline__ void halo_epilogue(const ConvHaloParams& p, uint32_t tmem_base, uint32_t acc_cols,
                                              uint64_t* acc_full, uint64_t* acc_empty, const float* s_scale,
                                              const float* s_shift, const float* s_headw, uint32_t stage_base,
                                              int warp, int lane) {
  constexpr int ESZ = fmt_esz(FMT);
  const int grp = warp & 3;                      // TMEM lane quarter
  const int egrp = (warp - 4) >> 2;              // epilogue group 0 / 1
  const int m = grp * 32 + lane;                 // accumulator row: pixel (m >> 3, m & 7) of each MMA tile
  const int nchunks = p.n_blk / CW;
  const int units = p.mt * nchunks;
  const bool dbg_nostore = BIU_DBG(p, 1);
  float hacc[kMaxHead];
#pragma unroll
  for (int h = 0; h < kMaxHead; ++h) hacc[h] = 0.f;
  // byte steps of one MMA tile (8 pixels along x) in the destination(s)
  const int j_bytes = (MODE == EPI_UP ? 16 : 8) * p.out_ctot * ESZ;
  const int jp_bytes = 4 * p.pool_ctot * ESZ;
  const int up_row_elems = 2 * p.W * p.out_ctot;                    // EPI_UP: one output row / plane, in elements
  const int up_plane_elems = 4 * p.H * p.W * p.out_ctot;
  // staged (transposed) stores: bf16, 32-channel chunks that land in ONE destination pixel per thread
  constexpr int LPP = 2 * ESZ;                   // 16-byte chunks per pixel of a 32-channel chunk
  const bool staged = CW == 32 && stage_base != 0 && p.out != nullptr && !dbg_nostore &&
                      (MODE == EPI_CONV || (MODE == EPI_UP && p.up_cout % 32 == 0));
  const uint32_t stage = staged ? stage_base + (uint32_t)(warp - 4) * (uint32_t)(32 * LPP * 16) : 0u;
  const int tr_px_bytes = (MODE == EPI_UP ? 2 : 1) * p.out_ctot * ESZ;
  const long long tr_row_bytes = (MODE == EPI_UP ? 2LL * up_row_elems : (long long)p.W * p.out_ctot) * ESZ;
  int it = 0;
  PROF_DECL(warp == 4 && lane == 0);
  for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ++it) {
    const HaloTile tl = halo_decode(p, t);
    const int as = it & 1;
    PROF_T0();
    mbar_wait(&acc_full[as], (it >> 1) & 1, 0x800 + as);
    PROF_ADD(8);
    tc_fence_after();
    const int px0 = tl.x0 + (m & 7), py = tl.y0 + (m >> 3);
    const bool row_ok = py < p.H;
    // this thread's pixel of MMA tile 0
    char* out0 = nullptr;
    char* pool0 = nullptr;
    if (MODE == EPI_UP) {
      const long long oplane = p.up_dims == 3 ? (long long)tl.b0 * (2 * p.D) + 2 * tl.z0 : (long long)tl.b0 * p.D + tl.z0;
      const long long opix = (oplane * (2 * p.H) + 2 * py) * (2 * p.W) + 2 * px0;
      out0 = reinterpret_cast<char*>(p.out) + (opix * p.out_ctot + p.out_coff) * ESZ;
    } else if (p.out != nullptr) {
      const long long pix = (((long long)tl.b0 * p.D + tl.z0) * p.H + py) * p.W + px0;
      out0 = reinterpret_cast<char*>(p.out) + (pix * p.out_ctot + p.out_coff + tl.n0) * ESZ;
    }
    if (POOL) {
      const long long ppix = (((long long)tl.b0 * p.D + tl.z0) * (p.H >> 1) + (py >> 1)) * (p.W >> 1) + (px0 >> 1);
      pool0 = reinterpret_cast<char*>(p.pool_out) + (ppix * p.pool_ctot + p.pool_coff + tl.n0) * ESZ;
    }
    // transposed view of the warp's 4 x 8 pixel group: this lane writes chunk (lane & 3) of pixel column lane >> 2
    char* tr0 = nullptr;
    uint32_t tr_rows = 0;
    if (staged) {
      const int ty = tl.y0 + grp * 4, tx = tl.x0 + lane / LPP;
      if (MODE == EPI_UP) {
        const long long oplane = p.up_dims == 3 ? (long long)tl.b0 * (2 * p.D) + 2 * tl.z0 : (long long)tl.b0 * p.D + tl.z0;
        const long long opix = (oplane * (2 * p.H) + 2 * ty) * (2 * p.W) + 2 * tx;
        tr0 = reinterpret_cast<char*>(p.out) + (opix * p.out_ctot + p.out_coff) * ESZ + (lane % LPP) * 16;
      } else {
        const long long pix = (((long long)tl.b0 * p.D + tl.z0) * p.H + ty) * p.W + tx;
        tr0 = reinterpret_cast<char*>(p.out) + (pix * p.out_ctot + p.out_coff + tl.n0) * ESZ + (lane % LPP) * 16;
      }
#pragma unroll
      for (int r = 0; r < 4; ++r) tr_rows |= (ty + r < p.H ? 1u : 0u) << r;
    }
    const bool pool_lane = (lane & 9) == 0;      // even x and even y
    const uint32_t trow = tmem_base + as * acc_cols + ((uint32_t)(grp * 32) << 16);
    const float* sc_n0 = s_scale + tl.n0;
    const float* sh_n0 = s_shift + tl.n0;

    // unit sequence of this warp. Plain: egrp, egrp + 2, ... Head: whole MMA tiles (runs of nchunks units).
    auto next_unit = [&](int u) -> int {
      if (MODE != EPI_HEAD) return u + 2;
      return ((u + 1) % nchunks != 0) ? u + 1 : u + 1 + nchunks;     // skip the other group's MMA tile
    };
    auto process = [&](int u, const uint32_t (&acc)[32]) {
      const int j = u / nchunks, c = u - j * nchunks;
      const bool ok = row_ok && (px0 + 8 * j) < p.W && !dbg_nostore;
      char* o = (ok && out0 != nullptr) ? out0 + j * j_bytes + (MODE == EPI_UP ? 0 : c * CW * ESZ) : nullptr;
      char* po = (POOL && ok && pool_lane) ? pool0 + j * jp_bytes + c * CW * ESZ : nullptr;
      char* tr = nullptr;
      uint32_t tr_mask = 0;
      if (staged) {
        const int xb = tl.x0 + 8 * j + lane / LPP;
        if (ESZ == 2) {
          tr_mask = xb < p.W ? tr_rows : 0u;
        } else {
#pragma unroll
          for (int r = 0; r < 8; ++r)
            tr_mask |= (((tr_rows >> (r >> 1)) & 1u) && (xb + (r & 1) * 4) < p.W) ? (1u << r) : 0u;
        }
      }
      if (staged && tr_mask != 0) {
        if (MODE == EPI_UP) {
          const int nn = tl.n0 + c * CW;
          const int qd = nn / p.up_cout, co = nn - qd * p.up_cout;
          tr = tr0 + j * j_bytes +
               (long long)((qd >> 2) * up_plane_elems + ((qd >> 1) & 1) * up_row_elems + (qd & 1) * p.out_ctot + co) * ESZ;
        } else {
          tr = tr0 + j * j_bytes + c * CW * ESZ;
        }
      }
      halo_epi_chunk<FMT, CW, MODE, POOL>(p, acc, sc_n0 + c * CW, sh_n0 + c * CW, s_headw + c * CW, o, po,
                                          tl.n0 + c * CW, hacc, up_plane_elems, up_row_elems, stage, tr, tr_row_bytes,
                                          tr_px_bytes, tr_mask, lane);
      if (MODE == EPI_HEAD && c == nchunks - 1) {
        if (row_ok && (px0 + 8 * j) < p.W) {
          const long long plane = (long long)p.D * p.H * p.W;
          const long long sp = ((long long)tl.z0 * p.H + py) * p.W + px0 + 8 * j;
#pragma unroll
          for (int h = 0; h < kMaxHead; ++h) {
            if (h >= p.head_n) break;
            const float val = apply_head_act(hacc[h] + __ldg(p.head_b + h), p.head_act[h]);
            const long long o2 = ((long long)tl.b0 * p.head_n + h) * plane + sp;
            if (p.out_val) p.out_val[o2] = val;
            if (p.out_u8) p.out_u8[o2] = (uint8_t)(val * 255.0f);     // unet/predict.py:200 truncating cast
          }
        }
#pragma unroll
        for (int h = 0; h < kMaxHead; ++h) hacc[h] = 0.f;
      }
    };
    int u = MODE == EPI_HEAD ? egrp * nchunks : egrp;
    if (BIU_DBG(p, 8)) u = units;
    uint32_t ra[32], rb2[32];
    PROF_T0();
    if (u < units) tmem_ld_cw<CW>(trow + u * CW, ra);
    while (u < units) {
      int un = next_unit(u);
      tmem_wait_regs<CW>(ra);
      if (un < units) tmem_ld_cw<CW>(trow + un * CW, rb2);
      process(u, ra);
      u = un;
      if (u >= units) break;
      un = next_unit(u);
      tmem_wait_regs<CW>(rb2);
      if (un < units) tmem_ld_cw<CW>(trow + un * CW, ra);
      process(u, rb2);
      u = un;
    }
    PROF_ADD(10);
    // this warp is done reading the accumulator stage: hand it back to the MMA issuer (CTA pairs: the leader's)
    tc_fence_before();
    __syncwarp();
    if (lane == 0) { if (CTA2) mbar_arrive_leader(&acc_empty[as]); else mbar_arrive(&acc_empty[as]); }
    PROF_ADD(11);
  }
}

template <int FMT, int KS, int MT, bool CTA2>
__global__ void __launch_bounds__(kHaloThreads, 1) conv_halo_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                    const __grid_constant__ CUtensorMap tmB,
                                                                    const ConvHaloParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t a_full[kMaxABufs], a_empty[kMaxABufs];
  __shared__ uint64_t b_full[kMaxBStages], b_empty[kMaxBStages];
  __shared__ uint64_t acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_slot;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const uint32_t smem_off = ((smem_u32(smem_raw) + 1023u) & ~1023u) - smem_u32(smem_raw);
  const uint32_t smem_base = smem_u32(smem_raw) + smem_off;
  const uint32_t b_base = smem_base + p.a_bufs * p.a_buf_bytes;
  float* s_scale =
      reinterpret_cast<float*>(smem_raw + smem_off + p.a_bufs * p.a_buf_bytes + p.b_stages * p.b_stage_bytes);
  float* s_shift = s_scale + p.n_total;
  float* s_headw = s_shift + p.n_total;
  // 8 x 2 KB staging tiles of the epilogue warps (0 when the plan reserved none)
  const uint32_t stage_base = p.stage_bytes ? ((smem_u32(s_headw + (p.mode == EPI_HEAD ? p.head_n * p.n_blk : 0)) + 15u) & ~15u) : 0u;
  const int pw = 8 * p.mt + 2 * p.halo;                          // smem tile pitch in pixels
  const int rows = 16 + 2 * p.halo;
  const uint32_t rb = p.row_bytes;
  const int taps_r = p.halo ? 3 * p.kd : 1;                      // (dz, dy) taps
  const int taps_x = p.halo ? 3 : 1;
  const uint32_t acc_cols = (uint32_t)(p.mt * p.n_blk);          // columns of one accumulator stage

  uint32_t ncols = 32;
  while (ncols < 2 * acc_cols) ncols <<= 1;

  for (int i = threadIdx.x; i < p.n_total; i += kHaloThreads) {
    s_scale[i] = p.scale[i];
    s_shift[i] = p.shift[i];
  }
  if (p.mode == EPI_HEAD)
    for (int i = threadIdx.x; i < p.head_n * p.n_blk; i += kHaloThreads) s_headw[i] = p.head_w[i];

  // CTA pairs: rank 0 of the cluster is the leader - it owns the "full" barriers both CTAs' TMA loads complete on and
  // the "accumulator drained" barrier both epilogues arrive on, and it issues the MMAs; the MMA completions are
  // multicast to the "empty" / "accumulator full" barriers of both CTAs.
  const uint32_t cta_rank = CTA2 ? cluster_ctarank() : 0u;
  const bool leader = cta_rank == 0u;
  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int i = 0; i < p.a_bufs; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int s = 0; s < p.b_stages; ++s) { mbar_init(&b_full[s], 1); mbar_init(&b_empty[s], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], CTA2 ? 16 : 8); }
    fence_mbar_init();
  }
  if (warp == 1) {
    if (CTA2) { tmem_alloc2(&tmem_slot, ncols); tmem_relinquish2(); }
    else { tmem_alloc(&tmem_slot, ncols); tmem_relinquish(); }
  }
  tc_fence_before();
  __syncthreads();
  if (CTA2) cluster_sync_all();                   // the peer's barriers are initialised before anything targets them
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  if (warp == 0) {
    // ================================== halo (A) producer ===================================
    if (elect_one()) {
      const uint32_t halo_tx = (uint32_t)(p.kd * rows * pw) * rb;
      int ab = 0;
      uint32_t aph = 0;
      PROF_DECL(true);
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        const HaloTile tl = halo_decode(p, t);
        for (int ch = 0; ch < p.cin_chunks; ++ch) {
          PROF_T0();
          mbar_wait(&a_empty[ab], aph ^ 1, 0x400 + ab);
          PROF_ADD(0);
          if (BIU_DBG(p, 4)) { mbar_arrive(&a_full[ab]); if (++ab == p.a_bufs) { ab = 0; aph ^= 1; } continue; }
          if (!CTA2) mbar_arrive_expect_tx(&a_full[ab], halo_tx);
          else if (leader) mbar_arrive_expect_tx(&a_full[ab], 2u * halo_tx);     // both CTAs' halo tiles land on this barrier
          // The tile is fetched as 2-row boxes issued back to back: one TMA operation keeps only a few dozen L2
          // requests in flight, many concurrent ones are needed to cover the L2 / HBM latency.
          const uint32_t box_bytes = 2u * (uint32_t)pw * rb;
          uint32_t dst = smem_base + ab * p.a_buf_bytes;
          for (int dz = 0; dz < p.kd; ++dz)
            for (int r2 = 0; r2 < rows / 2; ++r2, dst += box_bytes) {
              if (CTA2)
                asm volatile(
                    "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
                    "{%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
                    "l"(reinterpret_cast<uint64_t>(&tmA)), "r"(smem_u32(&a_full[ab]) & kPeerBitMask), "r"(ch * p.ck),
                    "r"(tl.x0 - p.halo), "r"(tl.y0 - p.halo + 2 * r2), "r"(tl.z0 - (p.kd >> 1) + dz), "r"(tl.b0)
                    : "memory");
              else
                asm volatile(
                    "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
                    "%5, %6, %7}], [%2];" ::"r"(dst),
                    "l"(reinterpret_cast<uint64_t>(&tmA)), "r"(smem_u32(&a_full[ab])), "r"(ch * p.ck),
                    "r"(tl.x0 - p.halo), "r"(tl.y0 - p.halo + 2 * r2), "r"(tl.z0 - (p.kd >> 1) + dz), "r"(tl.b0)
                    : "memory");
            }
          PROF_ADD(1);
          if (++ab == p.a_bufs) { ab = 0; aph ^= 1; }
        }
      }
    }
  } else if (warp == 2) {
    // ================================= weight (B) producer ==================================
    if (elect_one()) {
      const uint32_t b_tx = (uint32_t)(CTA2 ? p.n_blk / 2 : p.n_blk) * rb;      // CTA pairs: every CTA stages half of the rows
      const int n_half = CTA2 ? (int)cta_rank * (p.n_blk / 2) : 0;
      const int taps = taps_r * taps_x;
      int s = 0;
      uint32_t bph = 0;
      PROF_DECL(true);
      for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x) {
        if (p.b_resident && t != (int)blockIdx.x) break;
        const HaloTile tl = halo_decode(p, t);
        for (int ch = 0; ch < p.cin_chunks; ++ch)
          for (int tap = 0; tap < taps; ++tap) {
            PROF_T0();
            mbar_wait(&b_empty[s], bph ^ 1, 0x500 + s);
            PROF_ADD(2);
            if (BIU_DBG(p, 16)) { mbar_arrive(&b_full[s]); if (++s == p.b_stages) { s = 0; bph ^= 1; } continue; }
            if (CTA2) {
              if (leader) mbar_arrive_expect_tx(&b_full[s], 2u * b_tx);
              asm volatile(
                  "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, "
                  "{%3, %4, %5}], [%2];" ::"r"(b_base + s * p.b_stage_bytes),
                  "l"(reinterpret_cast<uint64_t>(&tmB)), "r"(smem_u32(&b_full[s]) & kPeerBitMask), "r"(ch * p.ck),
                  "r"(tl.n0 + n_half), "r"(tap)
                  : "memory");
            } else {
              mbar_arrive_expect_tx(&b_full[s], b_tx);
              asm volatile(
                  "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
                  "%5}], [%2];" ::"r"(b_base + s * p.b_stage_bytes),
                  "l"(reinterpret_cast<uint64_t>(&tmB)), "r"(smem_u32(&b_full[s])), "r"(ch * p.ck), "r"(tl.n0),
                  "r"(tap)
                  : "memory");
            }
            if (++s == p.b_stages) { s = 0; bph ^= 1; }
          }
      }
    }
  } else if (warp == 1 && leader) {
    // ====================================== MMA issuer ======================================
    // All 32 lanes run the loops (warp-uniform control flow and addresses); the elected lane issues. MT and KS are
    // compile-time so the MT*KS MMAs of a tap are straight-line code with immediate descriptor offsets.
    const bool issue = !BIU_DBG(p, 2);
    const uint32_t layout = rb == 128 ? 2u : (rb == 64 ? 4u : 6u);
    const uint32_t idesc = make_idesc(fmt_idesc(FMT), (uint32_t)p.n_blk, CTA2 ? 256u : 128u);
    // Descriptors: only the 14-bit start-address field (address >> 4) changes between MMAs and it never carries
    // out of the field (shared memory < 256 KB).
    const uint64_t a_desc0 = make_smem_desc(smem_base, (uint32_t)pw * rb, layout);
    const uint64_t b_desc0 = make_smem_desc(b_base, 8u * rb, layout);
    constexpr uint32_t j_step = 16u * KS;          // next MMA tile: 8 pixels further = 8 * row_bytes / 16
    constexpr uint32_t px_step = 2u * KS;          // one pixel
    const uint32_t row_step = ((uint32_t)pw * rb) >> 4;
    const uint32_t abuf_step = p.a_buf_bytes >> 4, bst_step = p.b_stage_bytes >> 4;
    const uint32_t n_blk = (uint32_t)p.n_blk;
    int ab = 0, bs = 0, it = 0;
    uint32_t aph = 0, bph = 0;
    PROF_DECL(lane == 0);
    for (int t = blockIdx.x; t < p.total_tiles; t += gridDim.x, ++it) {
      const int as = it & 1;
      PROF_T0();
      mbar_wait(&acc_empty[as], ((it >> 1) & 1) ^ 1, 0x900 + as);     // epilogue has drained this stage
      PROF_ADD(3);
      tc_fence_after();
      const uint32_t tacc = tmem_base + as * acc_cols;
      bool first = true;                                              // first k-block of a tile overwrites
      for (int ch = 0; ch < p.cin_chunks; ++ch) {
        PROF_T0();
        mbar_wait(&a_full[ab], aph, 0x600 + ab);
        PROF_ADD(4);
        const uint64_t a_buf_desc = a_desc0 + (uint64_t)(ab * abuf_step);
        for (int r = 0; r < taps_r; ++r) {                            // r = dz*3 + dy
          const int dz = r / 3, dy = r - 3 * dz;
          const uint64_t a_row_desc = a_buf_desc + (uint64_t)(BIU_DBG(p, 64) ? 0u : (uint32_t)(dz * rows + dy) * row_step);
          for (int dx = 0; dx < taps_x; ++dx) {
            PROF_T0();
            if (!p.b_resident || it == 0) {
              mbar_wait(&b_full[bs], bph, 0x700 + bs);
              tc_fence_after();
            }
            PROF_ADD(5);
            const uint64_t bd0 = b_desc0 + (uint64_t)(bs * bst_step);
            const uint64_t ad0 = a_row_desc + (uint64_t)(BIU_DBG(p, 64) ? 0u : dx * px_step);
            if (issue && elect_one()) {
              if (first) {
#pragma unroll
                for (int j = 0; j < MT; ++j)
#pragma unroll
                  for (int k = 0; k < KS; ++k) {
                    if (k == 0) tc_mma_imm<FMT, 0, CTA2>(tacc + j * n_blk, ad0 + (j * j_step + 2 * k), bd0 + 2 * k, idesc);
                    else tc_mma_imm<FMT, 1, CTA2>(tacc + j * n_blk, ad0 + (j * j_step + 2 * k), bd0 + 2 * k, idesc);
                  }
              } else {
#pragma unroll
                for (int j = 0; j < MT; ++j)
#pragma unroll
                  for (int k = 0; k < KS; ++k)
                    tc_mma_imm<FMT, 1, CTA2>(tacc + j * n_blk, ad0 + (j * j_step + 2 * k), bd0 + 2 * k, idesc);
              }
            }
            if (!p.b_resident && elect_one()) { if (CTA2) tc_commit2(&b_empty[bs]); else tc_commit(&b_empty[bs]); }
            first = false;
            PROF_ADD(6);
            if (++bs == p.b_stages) { bs = 0; bph ^= 1; }
          }
        }
        if (elect_one()) { if (CTA2) tc_commit2(&a_empty[ab]); else tc_commit(&a_empty[ab]); }
        if (++ab == p.a_bufs) { ab = 0; aph ^= 1; }
      }
      if (elect_one()) { if (CTA2) tc_commit2(&acc_full[as]); else tc_commit(&acc_full[as]); }
    }
  } else if (warp >= 4) {
    // ======================================= epilogue =======================================
#define BIU_EPI(CW, MODE, POOL) \
    halo_epilogue<FMT, CW, MODE, POOL, CTA2>(p, tmem_base, acc_cols, acc_full, acc_empty, s_scale, s_shift, s_headw, stage_base, warp, lane)
    if (p.n_blk % 32 == 0) {
      if (p.mode == EPI_CONV) { if (p.pool_out != nullptr) BIU_EPI(32, EPI_CONV, true); else BIU_EPI(32, EPI_CONV, false); }
      else if (p.mode == EPI_UP) BIU_EPI(32, EPI_UP, false);
      else BIU_EPI(32, EPI_HEAD, false);
    } else {
      if (p.mode == EPI_CONV) { if (p.pool_out != nullptr) BIU_EPI(16, EPI_CONV, true); else BIU_EPI(16, EPI_CONV, false); }
      else if (p.mode == EPI_UP) BIU_EPI(16, EPI_UP, false);
      else BIU_EPI(16, EPI_HEAD, false);
    }
#undef BIU_EPI
  }

  tc_fence_before();
  __syncthreads();
  if (CTA2) cluster_sync_all();       // the peer may still read this CTA's shared memory / signal its barriers
  if (warp == 1) { if (CTA2) tmem_dealloc2(tmem_base, ncols); else tmem_dealloc(tmem_base, ncols); }
}

#define BIU_HALO_LAUNCH(E, K, M)                                                                                  \
  do {                                                                                                             \
    if (p.cta2) {                                                                                                  \
      static int max_set2 = 0;                                                                                     \
      if (smem > max_set2) {                                                                                       \
        BIU_CHECK_CUDA(cudaFuncSetAttribute(conv_halo_kernel<E, K, M, true>,                                       \
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                   \
        max_set2 = smem;                                                                                           \
      }                                                                                                            \
      cudaLaunchConfig_t cfg;                                                                                      \
      memset(&cfg, 0, sizeof(cfg));                                                                                \
      cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kHaloThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream; \
      cudaLaunchAttribute at[1];                                                                                   \
      at[0].id = cudaLaunchAttributeClusterDimension;                                                              \
      at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;                          \
      cfg.attrs = at; cfg.numAttrs = 1;                                                                            \
      BIU_CHECK_CUDA(cudaLaunchKernelEx(&cfg, conv_halo_kernel<E, K, M, true>, tmA, tmB, p));                      \
    } else {                                                                                                       \
      static int max_set = 0;                                                                                      \
      if (smem > max_set) {                                                                                        \
        BIU_CHECK_CUDA(cudaFuncSetAttribute(conv_halo_kernel<E, K, M, false>,                                      \
                                            cudaFuncAttributeMaxDynamicSharedMemorySize, smem));                   \
        max_set = smem;                                                                                            \
      }                                                                                                            \
      conv_halo_kernel<E, K, M, false><<<grid, kHaloThreads, smem, stream>>>(tmA, tmB, p);                         \
    }                                                                                                              \
  } while (0)
#define BIU_HALO_LAUNCH_M(E, K)                                                                                    \
  do {                                                                                                             \
    if (p.mt == 8) BIU_HALO_LAUNCH(E, K, 8); else if (p.mt == 4) BIU_HALO_LAUNCH(E, K, 4);                          \
    else if (p.mt == 2) BIU_HALO_LAUNCH(E, K, 2); else BIU_HALO_LAUNCH(E, K, 1);                                    \
  } while (0)
// Host-side dispatch over the (k-steps per chunk, MMA tiles per work item) instantiations of one element format.
template <int FMT>
int halo_dispatch(const CUtensorMap& tmA, const CUtensorMap& tmB, const ConvHaloParams& p, int grid, int smem,
                  cudaStream_t stream) {
  const int ks = p.row_bytes / 32;
  if (ks == 4) BIU_HALO_LAUNCH_M(FMT, 4); else if (ks == 2) BIU_HALO_LAUNCH_M(FMT, 2); else BIU_HALO_LAUNCH_M(FMT, 1);
  return 0;
}

#define BIU_HALO_PAIRS(E, K, M)                                                                                    \
  do {                                                                                                             \
    if (cudaFuncSetAttribute(conv_halo_kernel<E, K, M, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != \
        cudaSuccess) { cudaGetLastError(); return 0; }                                                             \
    cudaLaunchConfig_t cfg;                                                                                        \
    memset(&cfg, 0, sizeof(cfg));                                                                                  \
    cfg.gridDim = dim3(2); cfg.blockDim = dim3(kHaloThreads); cfg.dynamicSmemBytes = smem;                         \
    cudaLaunchAttribute at[1];                                                                                     \
    at[0].id = cudaLaunchAttributeClusterDimension;                                                                \
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;                            \
    cfg.attrs = at; cfg.numAttrs = 1;                                                                              \
    int n = 0;                                                                                                     \
    if (cudaOccupancyMaxActiveClusters(&n, conv_halo_kernel<E, K, M, true>, &cfg) != cudaSuccess) {                \
      cudaGetLastError();                                                                                          \
      return 0;                                                                                                    \
    }                                                                                                              \
    return n;                                                                                                      \
  } while (0)
#define BIU_HALO_PAIRS_M(E, K)                                                                                     \
  do {                                                                                                             \
    if (mt == 8) BIU_HALO_PAIRS(E, K, 8); else if (mt == 4) BIU_HALO_PAIRS(E, K, 4);                                \
    else if (mt == 2) BIU_HALO_PAIRS(E, K, 2); else BIU_HALO_PAIRS(E, K, 1);                                        \
  } while (0)
// Co-resident CTA pairs of the 2-CTA kernel with `smem` bytes of dynamic shared memory (0: no cluster launch possible).
// The kernel is persistent with a static tile stride, so its grid must not exceed what is resident at once.
template <int FMT>
int halo_max_pairs(int ks, int mt, int smem) {
  if (ks == 4) BIU_HALO_PAIRS_M(FMT, 4); else if (ks == 2) BIU_HALO_PAIRS_M(FMT, 2); else BIU_HALO_PAIRS_M(FMT, 1);
  return 0;
}

// Each element format is instantiated in a translation unit of its own (conv_halo_bf16.cu / _f16.cu / _tf32.cu:
// BIU_HALO_INSTANCES(, FMT)), so that they compile in parallel; every other unit only declares them.
#define BIU_HALO_INSTANCES(EXTERN, E)                                                                                \
  EXTERN template int halo_dispatch<E>(const CUtensorMap&, const CUtensorMap&, const ConvHaloParams&, int, int,      \
                                       cudaStream_t);                                                                \
  EXTERN template int halo_max_pairs<E>(int, int, int);
BIU_HALO_INSTANCES(extern, FMT_BF16)
BIU_HALO_INSTANCES(extern, FMT_F16)
BIU_HALO_INSTANCES(extern, FMT_TF32)

}  // namespace biu
