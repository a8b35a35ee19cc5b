// Row-streaming 3x3(x3) convolution for NARROW layers (Cout <= 32; 2D bf16 / fp16 also Cout = 64) on tcgen05: the dy taps
// are folded into N.
//
// Why: with M = 128 the tensor core fetches its operands from shared memory at ~85 B/clk (measured,
// tools/conv_bench.cu): an MMA of N = 32 costs ~60 cycles for 16 cycles of math, so the 9-tap / 27-tap form of
// conv_halo.cuh is operand-fetch bound at ~25 % of the tensor peak for the full-resolution layers. Here one MMA
// multiplies an input row segment with the weights of all three dy taps at once (N = 3 * Cout):
//     E[r][x][dy, co] = sum_{dz, dx, ci} in[z + dz - 1][r][x + dx - 1][ci] * W[co][ci][dz][dy][dx]
//     out[y][x][co]   = E[y - 1][x][0, co] + E[y][x][1, co] + E[y + 1][x][2, co]
// i.e. 3 (x kd) MMAs of N = 96 per 16 input channels instead of 9 (x kd) of N = 32: ~2.1x fewer operand bytes per
// useful MAC. The epilogue adds the three partial rows while it drains TMEM.
//
// The three partial rows are summed by the tensor core itself: every OUTPUT row owns a TMEM slot of Cout fp32
// columns (ring of 512 / Cout = 16 or 32 slots, zeroed by the epilogue before reuse) and the MMA of input row r
// accumulates its N = 3*Cout result over the three consecutive slots of output rows r-1, r, r+1 (weights packed in
// the order dy = 2, 1, 0). Where the three slots wrap around the ring the MMA is split in two (N = Cout + 2*Cout).
// The deep ring lets the MMA warp run a dozen rows ahead of the epilogue: the kernel is no longer bound by the
// barrier round trips between the two (tools/conv_bench.cu: 600 cycles per row with a 5-slot ring of 3*Cout slots).
//
// Work item = a strip of 128 pixels (one MMA M tile = 128 consecutive x of one image row) x RB output rows of one
// plane. Input rows y0-1 .. y0+RB stream through a shared-memory ring (one TMA box of 130 pixels per row, plane and
// channel chunk; out-of-image rows / columns / planes are zero-filled = the convolution's padding). Per item the
// ring sees RB+4 "virtual" output rows: two dummies on either side collect the unused partial rows of the halo
// input rows and are only zeroed again. The folded weights of the layer stay resident in shared memory.
// (When a whole input row - all channel chunks - does not fit beside them, the ring's slots hold one channel chunk
// each: ConvRowsParams::cps.) Cout = 64: N = 192, eight TMEM slots of 64 columns, a row is drained in two halves.
// Warp roles: 0 = row (A) producer, 1 = TMEM alloc + MMA issuer (warp-uniform, see conv_halo.cuh), 2 = weight
// loader; with ConvRowsParams::pipes == 2 warps 2 and 3 are the producer and the MMA issuer of a SECOND, independent
// pipeline (own half of the A ring, of the TMEM slots and of the epilogue groups, alternate work items) that shares
// the resident weights and the tensor core - one issuing warp spends as long on a row's barrier bookkeeping as the
// tensor core on its six MMAs and the two do not overlap. 4..19 = epilogue: warp w drains TMEM lane quarter w % 4 (32 pixels, ALL channels) of every fourth PAIR of
// output rows (group (w - 4) / 4): four groups of four warps leapfrog over the row pairs, so one group's barrier wait /
// TMEM drain / slot zeroing overlaps the other groups' arithmetic and stores. A slot is released by the four arrivals
// of the group that drained it. Finished rows go through a per-warp, XOR-swizzled shared-memory tile and are written
// back transposed: consecutive lanes cover the consecutive 16-byte pieces of a pixel, so a warp store writes whole
// pixels (full 32-byte sectors, 512 contiguous bytes when the destination is dense) instead of 32 scattered 16-byte
// pieces - the same fix that took up4 from 1.70 to 0.93 ms in conv_halo.cuh. The 1x1 heads need no cross-warp
// combination any more (a thread holds all channels of its pixel).
#pragma once
#include "conv_halo.cuh"

namespace biu {

constexpr int kRowsMaxASlots = 24;
constexpr int kRowsMaxTSlots = 32;
constexpr int kRowsThreads = 640;
constexpr int kRowsPx = 130;                 // 128 pixels + 1 halo column on each side

struct ConvRowsParams {
  int W, H, D, B;
  int strips, rblocks, RB;       // strips of 128 px per row, row blocks per plane, rows per block
  int total_items;               // strips * rblocks * D * B
  int kd;                        // 1 (2D) or 3
  int cin_chunks, ck, row_bytes;
  int stage_px;                  // bytes of a pixel staged per epilogue pass (64, or 32 to save shared memory)
  int cps;                       // channel chunks per A-ring slot (cin_chunks, or 1 when a whole row does not fit)
  int cp;                        // padded output channels (16 or 32); N of the folded MMA = 3 * cp
  int a_slots;                   // shared-memory ring: one slot = one input row of one plane, all channel chunks
  uint32_t a_slot_bytes, a_chunk_bytes;
  uint32_t w_tile_bytes;         // one folded weight tile [(dy, co)][ck]; kd * 3 * cin_chunks of them
  int t_slots;                   // TMEM ring: 512 / cp slots of cp columns (one per output row)
  int pipes;                     // 1 or 2 independent pipelines (producer + MMA warp + epilogue groups) per CTA
  // PLANE mode (3D blocks on planes narrower than 128 px): the M tile is a 16 x 8 pixel tile of one plane, a ring slot
  // holds its 18 x 10 halo tile (all nine in-plane taps run out of it by row-shifted descriptors, as in conv_halo.cuh),
  // the dz taps are folded into N and the "rows" that stream through the TMEM slot ring are the PLANES z of the tile:
  // work item = tile x all D planes of one volume, weights packed [dy*3+dx][(2-dz)*cp + co][cin].
  int plane;
  int tiles_x, tiles_y;          // plane mode: 16 x 8 tiles per plane
  int slot_px;                   // pixels (shared-memory rows) per channel chunk of a slot: 130, or 18 * 10 = 180
  // K split over several launches (blocks whose resident weights would leave no room for the A ring, e.g. 96 input
  // channels x 27 taps): a launch covers the channel chunks [cin_chunk0, cin_chunk0 + cin_chunks) and
  //   acc_mode 1: stores its raw fp32 accumulators to acc_scratch [pixel][cp] instead of an output,
  //   acc_mode 3: adds the stored partial sums to its own and stores them again,
  //   acc_mode 2: adds them and finishes the block (BatchNorm, activation, store) as usual.   (0: single launch)
  int cin_chunk0;
  int acc_mode;
  float* acc_scratch;
  // FIRST mode (first block of the 2D nets, one uint8 input channel): the three dx taps are the K dimension. An A-ring row
  // is one pixel's {in[x-1], in[x], in[x+1], 0...} (32 bytes: bf16 / fp16 K = 16, tf32 K = 8) and is WRITTEN BY THE
  // PRODUCER WARP itself from the planar uint8 tile (integers 0..255 are exact in all three; the 1/255 of unet/predict.py:192 is
  // folded into the fp32 scale), so one MMA of N = 3 * Cout per input row does the whole block: w_taps = 1.
  int first;
  const uint8_t* first_in;       // [B][H][W] uint8
  int w_taps;                    // weight tiles per channel chunk: kd * 3, or 1 in first mode
  int mode;                      // EPI_CONV or EPI_HEAD
  float slope;
  const float* scale;
  const float* shift;
  void* out;
  int out_ctot, out_coff;
  void* pool_out;                // EPI_CONV, 2D: fused MaxPool2d(2) (may be null)
  int pool_ctot, pool_coff;
  int head_n;
  const float* head_w;           // [head_n][cp]
  const float* head_b;
  int head_act[kMaxHead];
  float* out_val;
  uint8_t* out_u8;
};

template <int HC>
__device__ __forceinline__ void tmem_ld_hc(uint32_t taddr, uint32_t (&r)[16]) {
  if (HC == 16) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "
        "%15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
  } else {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
  }
}
template <int HC>
__device__ __forceinline__ void tmem_wait3(uint32_t (&a)[16], uint32_t (&b)[16], uint32_t (&c)[16]) {
  if (HC == 16) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                   "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                   "+r"(b[8]), "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15]),
                   "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]), "+r"(c[4]), "+r"(c[5]), "+r"(c[6]), "+r"(c[7]),
                   "+r"(c[8]), "+r"(c[9]), "+r"(c[10]), "+r"(c[11]), "+r"(c[12]), "+r"(c[13]), "+r"(c[14]), "+r"(c[15])
                 :
                 : "memory");
  } else {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]),
                   "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3]), "+r"(c[4]), "+r"(c[5]), "+r"(c[6]), "+r"(c[7])
                 :
                 : "memory");
  }
}

template <int HC>
__device__ __forceinline__ void tmem_wait1(uint32_t (&a)[16]) {
  if (HC == 16) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15])
                 :
                 : "memory");
  } else {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7])
                 :
                 : "memory");
  }
}
// zero HC consecutive fp32 columns of this warp's 32 TMEM lanes
template <int HC>
__device__ __forceinline__ void tmem_zero_hc(uint32_t taddr) {
  const uint32_t z = 0;
  if (HC == 16) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
        ::"r"(taddr), "r"(z) : "memory");
  } else {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z)
                 : "memory");
  }
}
// CP consecutive fp32 columns (16 or 32) of this warp's 32 TMEM lanes
template <int CP>
__device__ __forceinline__ void tmem_ld_cp(uint32_t taddr, uint32_t (&r)[CP]) {
  if (CP == 32) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16 % CP]), "=r"(r[17 % CP]), "=r"(r[18 % CP]), "=r"(r[19 % CP]), "=r"(r[20 % CP]), "=r"(r[21 % CP]),
          "=r"(r[22 % CP]), "=r"(r[23 % CP]), "=r"(r[24 % CP]), "=r"(r[25 % CP]), "=r"(r[26 % CP]), "=r"(r[27 % CP]),
          "=r"(r[28 % CP]), "=r"(r[29 % CP]), "=r"(r[30 % CP]), "=r"(r[31 % CP])
        : "r"(taddr)
        : "memory");
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
template <int CP>
__device__ __forceinline__ void tmem_ld_wait_cp(uint32_t (&a)[CP]) {
  if (CP == 32) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]),
                   "+r"(a[16 % CP]), "+r"(a[17 % CP]), "+r"(a[18 % CP]), "+r"(a[19 % CP]), "+r"(a[20 % CP]),
                   "+r"(a[21 % CP]), "+r"(a[22 % CP]), "+r"(a[23 % CP]), "+r"(a[24 % CP]), "+r"(a[25 % CP]),
                   "+r"(a[26 % CP]), "+r"(a[27 % CP]), "+r"(a[28 % CP]), "+r"(a[29 % CP]), "+r"(a[30 % CP]),
                   "+r"(a[31 % CP])
                 :
                 : "memory");
  } else {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]),
                   "+r"(a[8]), "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15])
                 :
                 : "memory");
  }
}
template <int CP>
__device__ __forceinline__ void tmem_zero_cp(uint32_t taddr) {
  const uint32_t z = 0;
#pragma unroll
  for (int c = 0; c < CP; c += 16)
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};"
        ::"r"(taddr + (uint32_t)c), "r"(z) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

#ifdef BIU_DBG_KNOBS
static __device__ int g_rows_dbg = 0;
#endif

struct RowsItem { int x0, y0, rows, z, b; };

__device__ __forceinline__ RowsItem rows_decode(const ConvRowsParams& p, int t) {
  RowsItem r;
  if (p.plane) {
    const int tx = t % p.tiles_x; t /= p.tiles_x;
    const int ty = t % p.tiles_y; t /= p.tiles_y;
    r.b = t; r.z = 0; r.x0 = tx * 8; r.y0 = ty * 16; r.rows = p.D;
    return r;
  }
  const int sx = t % p.strips; t /= p.strips;
  const int rb = t % p.rblocks; t /= p.rblocks;
  r.z = t % p.D; t /= p.D;
  r.b = t;
  r.x0 = sx * 128;
  r.y0 = rb * p.RB;
  r.rows = min(p.RB, p.H - r.y0);
  return r;
}

// Epilogue of all work items for one warp. CP = padded output channels (all of them are handled by this warp).
template <int FMT, int CP, int MODE, bool POOL, int SBW = 64>
__device__ __forceinline__ void rows_epilogue(const ConvRowsParams& p, uint32_t tmem_base, uint64_t* t_full,
                                              uint64_t* t_empty, const float* s_scale, const float* s_shift,
                                              const float* s_headw, uint8_t* stage, int warp, int lane) {
  constexpr int ESZ = fmt_esz(FMT);
  constexpr int PXB = CP * ESZ;                  // bytes of one output pixel
  constexpr int HC = CP > 32 ? 32 : CP;          // TMEM columns per drain (64-channel rows are drained in two halves)
  constexpr int NH = CP / HC;
  constexpr int NW = PXB / 4;                    // 32-bit words per pixel
  constexpr int NV = PXB / 16;                   // 16-byte pieces per pixel: 2, 4 or 8
  constexpr int SB = PXB < SBW ? PXB : SBW;      // bytes of a pixel staged per pass (wider pixels go in several passes; SBW = 32
                                                 // keeps the tiles small when a 64-channel block's weights need the room)
  constexpr int SV = SB / 16;                    // 16-byte pieces per pixel and pass: 2 or 4
  constexpr int PASSES = PXB / SB;
  constexpr int PPI = 32 / SV;                   // pixels covered by one transposed warp store
  const int q = warp & 3;                        // TMEM lane quarter: pixels 32q .. 32q+31 of the strip
  const int grp = (warp - 4) >> 2;               // 0..3
  const int gpp = 4 / p.pipes;                   // epilogue groups per pipeline
  const int pipe = grp / gpp, gi = grp - pipe * gpp;   // this warp's row pairs: running pair count % gpp == gi
  const int tsl = p.t_slots / p.pipes;           // TMEM ring of this pipeline: slots [pipe * tsl, (pipe + 1) * tsl)
  const int slot0 = pipe * tsl;
  const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
  const int lg_slots = tsl == 32 ? 5 : (tsl == 16 ? 4 : 3);
  int ts = 0;                                    // ring position (slot + tsl * use parity) of the item's first virtual row
  int gcnt = 0;                                  // number of row pairs of the earlier items, mod gpp
  // staging tile of this warp: [32 pixels][SB bytes], 16-byte pieces XOR-swizzled so that both the per-pixel writes
  // and the transposed reads are bank-conflict free
  uint8_t* tile = stage + (size_t)(warp - 4) * (32 * SB);
  const int wr_swz = SV == 4 ? ((lane >> 1) & 3) : ((lane >> 2) & 1);
  const int rd_piece = lane % SV, rd_px = lane / SV;

  // Before anything accumulates: zero every slot and mark all slots empty (phase 0) - the first group of a pipeline
  // does it for the pipeline.
  if (gi == 0) {
    for (int sl = slot0; sl < slot0 + tsl; ++sl) tmem_zero_cp<CP>(tmem_base + lane_addr + (uint32_t)(sl * CP));
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0)
      for (int sl = slot0; sl < slot0 + tsl; ++sl) mbar_arrive(&t_empty[sl]);
  }

  for (int t = blockIdx.x + pipe * gridDim.x; t < p.total_items; t += p.pipes * gridDim.x) {
    const RowsItem it = rows_decode(p, t);
    // row mode: the quarter = 32 consecutive pixels of the strip; plane mode: rows 4q .. 4q+3 of the 16 x 8 tile
    const bool plane = p.plane != 0;
    const int px0 = plane ? it.x0 : it.x0 + q * 32;     // first pixel (column) of this warp's quarter
    const int px = px0 + lane;
#ifdef BIU_DBG_KNOBS
    const int npix = (g_rows_dbg & 8) ? 0 : min(32, p.W - px0);
#else
    const int npix = min(32, p.W - px0);         // row mode: valid pixels of the quarter (<= 0: none)
#endif
    const int q_rows = plane ? min(4, p.H - (it.y0 + 4 * q)) : 0, q_cols = plane ? min(8, p.W - it.x0) : 0;
    auto pix_ok = [&](int pxi) { return plane ? ((pxi >> 3) < q_rows && (pxi & 7) < q_cols) : pxi < npix; };
    const bool col_ok = pix_ok(lane);
    const long long plane_row0 = ((long long)it.b * p.D + it.z) * p.H + it.y0 + (plane ? 4 * q : 0);
    char* out_q = nullptr;                       // first pixel of the quarter in the item's first output row / plane
    if (MODE == EPI_CONV)
      out_q = reinterpret_cast<char*>(p.out) + ((plane_row0 * p.W + px0) * p.out_ctot + p.out_coff) * ESZ;
    const long long out_row_bytes = (plane ? (long long)p.H * p.W : (long long)p.W) * p.out_ctot * ESZ;   // next output row / plane
    const int out_px_bytes = p.out_ctot * ESZ;
    const long long out_q8_bytes = (plane ? (long long)p.W : 8LL) * out_px_bytes;      // 8 quarter-pixels further
    const int st_lane_off = (int)((rd_px >> 3) * out_q8_bytes) + (rd_px & 7) * out_px_bytes + rd_piece * 16;
    const int rd_lane_off = rd_px * SB + ((rd_piece ^ (SV == 4 ? ((rd_px >> 1) & 3) : ((rd_px >> 2) & 1))) << 4);
    // K split: this lane's pixel in the fp32 partial-sum scratch [pixel][CP] (pixel index of output row / plane o = + o * pix_per_o)
    const long long lane_pix0 = plane ? (plane_row0 + (lane >> 3)) * p.W + px0 + (lane & 7) : plane_row0 * p.W + px;
    const long long pix_per_o = plane ? (long long)p.H * p.W : (long long)p.W;
    auto partial = [&](uint32_t (&e)[HC], int o, int hh, int mode) {        // mode bit 1: add the stored sums, bit 0: store
      if (!col_ok) return;
      float4* sp = reinterpret_cast<float4*>(p.acc_scratch + (lane_pix0 + o * pix_per_o) * CP + hh * HC);
      if (mode & 2) {
#pragma unroll
        for (int i4 = 0; i4 < HC / 4; ++i4) {
          const float4 s4 = sp[i4];
          e[4 * i4 + 0] = __float_as_uint(__uint_as_float(e[4 * i4 + 0]) + s4.x);
          e[4 * i4 + 1] = __float_as_uint(__uint_as_float(e[4 * i4 + 1]) + s4.y);
          e[4 * i4 + 2] = __float_as_uint(__uint_as_float(e[4 * i4 + 2]) + s4.z);
          e[4 * i4 + 3] = __float_as_uint(__uint_as_float(e[4 * i4 + 3]) + s4.w);
        }
      }
      if (mode & 1) {
#pragma unroll
        for (int i4 = 0; i4 < HC / 4; ++i4)
          sp[i4] = make_float4(__uint_as_float(e[4 * i4 + 0]), __uint_as_float(e[4 * i4 + 1]),
                               __uint_as_float(e[4 * i4 + 2]), __uint_as_float(e[4 * i4 + 3]));
      }
    };
    const int amode = (MODE == EPI_CONV && !POOL) ? p.acc_mode : 0;
    const bool finish = !(amode & 1);              // this launch produces the block's output
    char* pool_px = nullptr;
    long long pool_row_bytes = 0;
    if (POOL && !plane) {
      const long long prow0 = ((long long)it.b * p.D + it.z) * (p.H >> 1) + (it.y0 >> 1);
      pool_px = reinterpret_cast<char*>(p.pool_out) + ((prow0 * (p.W >> 1) + (px >> 1)) * p.pool_ctot + p.pool_coff) * ESZ;
      pool_row_bytes = (long long)(p.W >> 1) * p.pool_ctot * ESZ;
    } else if (POOL) {
      // plane mode = MaxPool3d(2): the row pairs below are PLANE pairs (z), the (y, x) pairs lie inside the warp's 4 x 8
      // pixels (lanes ^ 8 and ^ 1); pool_px = this lane's pooled pixel in pooled plane 0, one pooled plane per pair
      const long long prow0 = ((long long)it.b * (p.D >> 1)) * (p.H >> 1) + ((it.y0 + 4 * q + (lane >> 3)) >> 1);
      pool_px = reinterpret_cast<char*>(p.pool_out) +
                ((prow0 * (p.W >> 1) + ((it.x0 + (lane & 7)) >> 1)) * p.pool_ctot + p.pool_coff) * ESZ;
      pool_row_bytes = (long long)(p.H >> 1) * (p.W >> 1) * p.pool_ctot * ESZ;
    }
    const int vrows = it.rows + 4;               // virtual output rows: 2 dummies, rows real ones, 2 dummies

    const unsigned long long slope2 = pack_f32x2(p.slope, p.slope);
    // BatchNorm + LeakyReLU of one drained row, packed in the storage format (bf16 / fp16 pairs, tf32-rounded floats)
    auto activate = [&](const uint32_t (&e)[HC], uint32_t (&w)[NW], int hh) {     // channels hh * HC .. hh * HC + HC - 1
      constexpr int NWH = HC * ESZ / 4;
#pragma unroll
      for (int i4 = 0; i4 < HC / 4; ++i4) {
        // packed pairs (FFMA2 / FMUL2): two IEEE operations per issue slot, bit-identical to fmaf / a * slope - the
        // epilogue warps are issue-bound at full resolution
        const ulonglong2 sc = reinterpret_cast<const ulonglong2*>(s_scale + hh * HC)[i4];
        const ulonglong2 sh = reinterpret_cast<const ulonglong2*>(s_shift + hh * HC)[i4];
        const unsigned long long t0 = fma_f32x2(pack_f32x2(__uint_as_float(e[4 * i4]), __uint_as_float(e[4 * i4 + 1])), sc.x, sh.x);
        const unsigned long long t1 = fma_f32x2(pack_f32x2(__uint_as_float(e[4 * i4 + 2]), __uint_as_float(e[4 * i4 + 3])), sc.y, sh.y);
        const unsigned long long u0 = mul_f32x2(t0, slope2), u1 = mul_f32x2(t1, slope2);
        float a[4], u[4];
        unpack_f32x2(t0, a[0], a[1]); unpack_f32x2(t1, a[2], a[3]);
        unpack_f32x2(u0, u[0], u[1]); unpack_f32x2(u1, u[2], u[3]);
#pragma unroll
        for (int k = 0; k < 4; ++k) a[k] = fmaxf(a[k], u[k]);        // LeakyReLU for 0 <= slope <= 1
        if (ESZ == 2) {
          w[(hh * NWH + 2 * i4) % NW] = pack_half2<FMT>(a[0], a[1]);
          w[(hh * NWH + 2 * i4 + 1) % NW] = pack_half2<FMT>(a[2], a[3]);
        } else {
#pragma unroll
          for (int k = 0; k < 4; ++k) w[(hh * NWH + 4 * i4 + k) % NW] = __float_as_uint(round_tf32(a[k]));
        }
      }
    };
    // real output row o: through the staging tile, transposed, to global memory
    auto emit = [&](const uint32_t (&w)[NW], int o) {
#pragma unroll
      for (int h = 0; h < PASSES; ++h) {
        __syncwarp();                              // the previous transposed reads are done
#pragma unroll
        for (int j = 0; j < SV; ++j)
          *reinterpret_cast<uint4*>(tile + lane * SB + ((j ^ wr_swz) << 4)) =
              make_uint4(w[4 * (h * SV + j)], w[4 * (h * SV + j) + 1], w[4 * (h * SV + j) + 2], w[4 * (h * SV + j) + 3]);
        __syncwarp();
        // pixel i * PPI + rd_px: PPI is 8 or 16, so consecutive i are whole quarter-rows apart and the swizzle term and
        // the position inside the quarter-row depend on the lane only - one pointer per row, constant steps per store
        char* optr = out_q + o * out_row_bytes + h * SV * 16 + st_lane_off;
        const uint8_t* tptr = tile + rd_lane_off;
#pragma unroll
        for (int i = 0; i < SV; ++i) {
          const uint4 v4 = *reinterpret_cast<const uint4*>(tptr + i * (PPI * SB));
          if (pix_ok(i * PPI + rd_px)) *reinterpret_cast<uint4*>(optr + i * (PPI / 8) * out_q8_bytes) = v4;
        }
      }
    };
    // 1x1 heads of real output row o (a thread holds every channel of its pixel)
    auto heads = [&](uint32_t (&e)[HC], int o) {     // MODE == EPI_HEAD is only instantiated for CP <= 32 (HC == CP)
      float hacc[kMaxHead];
#pragma unroll
      for (int i4 = 0; i4 < HC / 4; ++i4) {          // activation in place
        const float4 sc = reinterpret_cast<const float4*>(s_scale)[i4];
        const float4 sh = reinterpret_cast<const float4*>(s_shift)[i4];
        const float scv[4] = {sc.x, sc.y, sc.z, sc.w}, shv[4] = {sh.x, sh.y, sh.z, sh.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          float a = fmaf(__uint_as_float(e[4 * i4 + k]), scv[k], shv[k]);
          a = fmaxf(a, a * p.slope);
          if (ESZ == 4) a = round_tf32(a);
          e[4 * i4 + k] = __float_as_uint(a);
        }
      }
#pragma unroll
      for (int h = 0; h < kMaxHead; ++h) {
        if (h >= p.head_n) break;
        float s0 = 0.f, s1 = 0.f;
#pragma unroll
        for (int i4 = 0; i4 < HC / 4; ++i4) {
          const float4 hw = reinterpret_cast<const float4*>(s_headw + h * CP)[i4];
          s0 = fmaf(__uint_as_float(e[4 * i4]), hw.x, s0);
          s1 = fmaf(__uint_as_float(e[4 * i4 + 1]), hw.y, s1);
          s0 = fmaf(__uint_as_float(e[4 * i4 + 2]), hw.z, s0);
          s1 = fmaf(__uint_as_float(e[4 * i4 + 3]), hw.w, s1);
        }
        hacc[h] = s0 + s1;
      }
      if (col_ok) {
        const long long plane = (long long)p.D * p.H * p.W;
        // row mode: output row o of plane it.z; plane mode: this lane's pixel of the 16 x 8 tile in output plane o
        const long long sp = p.plane ? ((long long)o * p.H + it.y0 + 4 * q + (lane >> 3)) * p.W + it.x0 + (lane & 7)
                                     : ((long long)it.z * p.H + it.y0 + o) * p.W + px;
#pragma unroll
        for (int h = 0; h < kMaxHead; ++h) {
          if (h >= p.head_n) break;
          const float val = apply_head_act(hacc[h] + __ldg(p.head_b + h), p.head_act[h]);
          const long long o2 = ((long long)it.b * p.head_n + h) * plane + sp;
          if (p.out_val) p.out_val[o2] = val;
          if (p.out_u8) p.out_u8[o2] = (uint8_t)(val * 255.0f);     // unet/predict.py:200 truncating cast
        }
      }
    };

    // Virtual rows are handled in PAIRS (one barrier wait and one zero-store wait per two rows): wait until the later
    // row has all its partial rows, drain both (real rows only), zero both slots for their next users and release
    // them, then finish the arithmetic and the stores while the other groups are already at the next pairs.
    auto is_real = [&](int v) { return v >= 2 && v < it.rows + 2; };
    const int npairs = (vrows + 1) >> 1;
    for (int k = (gi - gcnt) & (gpp - 1); k < npairs; k += gpp) {
      const int v = 2 * k;
      const bool two = v + 1 < vrows;
      const int r0 = ts + v, r1 = r0 + 1;
      const int sl = slot0 + (r0 & (tsl - 1)), s1 = slot0 + (r1 & (tsl - 1));
      const uint32_t ph = (uint32_t)(r0 >> lg_slots) & 1u, p1 = (uint32_t)(r1 >> lg_slots) & 1u;
      if (two) mbar_wait(&t_full[s1], p1, 0xA00 + s1);                       // rows complete in order
      else mbar_wait(&t_full[sl], ph, 0xA00 + sl);
      tc_fence_after();
      const bool real0 = is_real(v), real1 = two && is_real(v + 1);
#ifdef BIU_DBG_KNOBS
      const bool drain = !(g_rows_dbg & 2);
#else
      const bool drain = true;
#endif
      uint32_t acc[HC];
      uint32_t w0[NW], w1[NW];
      if (real0) {
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
          if (drain) tmem_ld_cp<HC>(tmem_base + lane_addr + (uint32_t)(sl * CP + hh * HC), acc);
          tmem_ld_wait_cp<HC>(acc);
          if (MODE == EPI_HEAD) heads(acc, v - 2);
          else {
            if (amode) partial(acc, v - 2, hh, amode);
            if (finish) activate(acc, w0, hh);
          }
        }
      }
      if (real1) {
#pragma unroll
        for (int hh = 0; hh < NH; ++hh) {
          if (drain) tmem_ld_cp<HC>(tmem_base + lane_addr + (uint32_t)(s1 * CP + hh * HC), acc);
          tmem_ld_wait_cp<HC>(acc);
          if (NH > 1) {                             // 64-channel rows: activated half by half before the release
            if (amode) partial(acc, v - 1, hh, amode);
            if (finish) activate(acc, w1, hh);
          }
        }
      }
      tmem_zero_cp<CP>(tmem_base + lane_addr + (uint32_t)(sl * CP));
      if (two) tmem_zero_cp<CP>(tmem_base + lane_addr + (uint32_t)(s1 * CP));
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) { mbar_arrive(&t_empty[sl]); if (two) mbar_arrive(&t_empty[s1]); }
#ifdef BIU_DBG_KNOBS
      if (g_rows_dbg & 64) continue;
#endif
      if (MODE == EPI_HEAD) {
        if (real1) heads(acc, v - 1);
      } else {
        if (real0 && finish) emit(w0, v - 2);      // before row 1 is activated: keeps the live registers at two rows
        if (real1) {
          if (NH == 1) {
            if (amode) partial(acc, v - 1, 0, amode);
            if (finish) activate(acc, w1, 0);
          }
          if (finish) emit(w1, v - 1);
        }
        if (POOL && real0 && real1) {              // MaxPool2d(2): x pairs are adjacent lanes, y pairs = this row pair
          if (ESZ == 2) {                          // (plane mode, MaxPool3d(2): the pair is a z pair, y pairs are lanes ^ 8)
#pragma unroll
            for (int i = 0; i < NW; ++i) {
              uint32_t mx = max_half2<FMT>(w0[i], w1[i]);
              mx = max_half2<FMT>(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
              if (plane) mx = max_half2<FMT>(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
              w0[i] = mx;
            }
          } else {
#pragma unroll
            for (int i = 0; i < NW; ++i) {
              float mx = fmaxf(__uint_as_float(w0[i]), __uint_as_float(w1[i]));
              mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
              if (plane) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 8));
              w0[i] = __float_as_uint(mx);
            }
          }
          if (col_ok && !(lane & (plane ? 9 : 1))) {
            uint4* d4 = reinterpret_cast<uint4*>(pool_px + ((v - 2) >> 1) * pool_row_bytes);
#pragma unroll
            for (int j = 0; j < NV; ++j) d4[j] = make_uint4(w0[4 * j], w0[4 * j + 1], w0[4 * j + 2], w0[4 * j + 3]);
          }
        }
      }
    }
    ts = (ts + vrows) & (2 * tsl - 1);
    gcnt = (gcnt + npairs) & (gpp - 1);
  }
}

template <int FMT, int KS>
__global__ void __launch_bounds__(kRowsThreads, 1) conv_rows_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                    const __grid_constant__ CUtensorMap tmW,
                                                                    const ConvRowsParams p) {
  constexpr int ESZ = fmt_esz(FMT);
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint64_t a_full[kRowsMaxASlots], a_empty[kRowsMaxASlots];
  __shared__ uint64_t t_full[kRowsMaxTSlots], t_empty[kRowsMaxTSlots];
  __shared__ uint64_t w_full;
  __shared__ uint32_t tmem_slot;

  const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0);   // warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const uint32_t smem_off = ((smem_u32(smem_raw) + 1023u) & ~1023u) - smem_u32(smem_raw);
  const uint32_t smem_base = smem_u32(smem_raw) + smem_off;
  const int w_tiles = p.w_taps * p.cin_chunks;
  const uint32_t a_base = smem_base + (uint32_t)w_tiles * p.w_tile_bytes;
  uint8_t* tail = smem_raw + smem_off + (size_t)w_tiles * p.w_tile_bytes + (size_t)p.a_slots * p.a_slot_bytes;
  float* s_scale = reinterpret_cast<float*>(tail);
  float* s_shift = s_scale + p.cp;
  float* s_headw = s_shift + p.cp;                        // [head_n][cp]
  uint8_t* stage = reinterpret_cast<uint8_t*>(s_headw + kMaxHead * p.cp);   // 16 warps x [32 px][min(cp * ESZ, 64) bytes]
  const uint32_t rb = p.row_bytes;
  const int nfold = 3 * p.cp;

  for (int i = threadIdx.x; i < p.cp; i += kRowsThreads) { s_scale[i] = p.scale[i]; s_shift[i] = p.shift[i]; }
  if (p.mode == EPI_HEAD)
    for (int i = threadIdx.x; i < p.head_n * p.cp; i += kRowsThreads) s_headw[i] = p.head_w[i];

  if (warp == 0 && elect_one()) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmW);
    for (int i = 0; i < p.a_slots; ++i) { mbar_init(&a_full[i], 1); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < p.t_slots; ++i) { mbar_init(&t_full[i], 1); mbar_init(&t_empty[i], 4); }
    mbar_init(&w_full, 1);
    fence_mbar_init();
  }
  if (warp == 1) {
    tmem_alloc(&tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;

  // Two independent pipelines (p.pipes == 2) share the resident weights and the tensor core: pipeline 0 = producer
  // warp 0 + MMA warp 1, pipeline 1 = producer warp 2 + MMA warp 3, each with its own half of the A ring, of the TMEM
  // slot ring and of the epilogue groups, working on alternate items. While one MMA warp is busy with its barrier
  // bookkeeping the other one's MMAs keep the tensor core fed (a single issuing warp spends about as long on the
  // bookkeeping of a 6-MMA row as the tensor core on its MMAs, and the two do not overlap - tools/conv_bench.cu).
  const int pipes = p.pipes;
  const int asl = p.a_slots / pipes, tsl = p.t_slots / pipes;
  if (warp == 2) {
    // ============================ folded weights: loaded once, resident ============================
    if (elect_one()) {
      mbar_arrive_expect_tx(&w_full, (uint32_t)w_tiles * (uint32_t)nfold * rb);
      for (int tdx = 0; tdx < p.w_taps; ++tdx)                     // tdx = dz * 3 + dx
        for (int ch = 0; ch < p.cin_chunks; ++ch)
          asm volatile(
              "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
              "%5}], [%2];" ::"r"(smem_base + (uint32_t)(tdx * p.cin_chunks + ch) * p.w_tile_bytes),
              "l"(reinterpret_cast<uint64_t>(&tmW)), "r"(smem_u32(&w_full)), "r"((p.cin_chunk0 + ch) * p.ck), "r"(0), "r"(tdx)
              : "memory");
    }
  }
  if (p.first && (warp == 0 || (warp == 2 && pipes == 2))) {
    // ===================== first block: the producer warp builds the A rows itself =====================
    const int pipe = warp >> 1;
    const int a0 = pipe * asl;
    uint8_t* ring = smem_raw + smem_off + (size_t)w_tiles * p.w_tile_bytes + (size_t)a0 * p.a_slot_bytes;
    for (uint32_t i = lane; i < (uint32_t)asl * p.a_slot_bytes / 16; i += 32)       // K padding stays zero for good
      reinterpret_cast<uint4*>(ring)[i] = make_uint4(0, 0, 0, 0);
    __syncwarp();
    int as = 0;
    uint32_t aph = 0;
    for (int t = blockIdx.x + pipe * gridDim.x; t < p.total_items; t += pipes * gridDim.x) {
      const RowsItem it = rows_decode(p, t);
      const uint8_t* img = p.first_in + (long long)it.b * p.H * p.W;
      const int xb = it.x0 + 4 * lane;                           // this lane's four pixels xb .. xb + 3
      // One aligned 32-bit load per lane and row (pixels xb .. xb + 3; lane 0 / 31 also fetch the strip's two halo pixels),
      // issued TWO row pairs ahead of their use: the warp handles the rows one after the other, so an exposed global-memory
      // round trip per row would bound the whole kernel. The neighbours' edge pixels come by shuffle.
      const bool vec = (p.W & 3) == 0 && ((reinterpret_cast<uintptr_t>(img) & 3) == 0);
      auto fetch = [&](int i, uint32_t& w, uint32_t& edge) {      // edge: x = it.x0 - 1 (lane 0) / it.x0 + 128 (lane 31)
        const int y = it.y0 - 1 + i;
        w = 0; edge = 0;
        if (y < 0 || y >= p.H || i >= it.rows + 2) return;
        const uint8_t* row = img + (long long)y * p.W;
        if (vec) {
          if (xb < p.W) w = __ldg(reinterpret_cast<const uint32_t*>(row + xb));
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (xb + j < p.W) w |= (uint32_t)__ldg(row + xb + j) << (8 * j);
        }
        const int xe = lane == 0 ? it.x0 - 1 : it.x0 + 128;
        if ((lane == 0 || lane == 31) && xe >= 0 && xe < p.W) edge = __ldg(row + xe);
      };
      // one input row into its ring slot: row r = pixel it.x0 + r = {in[x-1], in[x], in[x+1], 0...}
      auto put = [&](uint32_t w, uint32_t edge, uint8_t* slot) {
        const uint32_t up = __shfl_up_sync(0xffffffffu, w, 1), dn = __shfl_down_sync(0xffffffffu, w, 1);
        float v[6];
        v[0] = (float)(lane == 0 ? edge : (up >> 24));
        v[1] = (float)(w & 0xffu); v[2] = (float)((w >> 8) & 0xffu); v[3] = (float)((w >> 16) & 0xffu); v[4] = (float)(w >> 24);
        v[5] = (float)(lane == 31 ? edge : (dn & 0xffu));
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = 4 * lane + j;                             // 32B swizzle: 16-byte chunk ^ ((r >> 2) & 1)
          uint8_t* row = slot + r * 32 + (((r >> 2) & 1) << 4);
          if (ESZ == 2) {
            *reinterpret_cast<uint2*>(row) = make_uint2(pack_half2<FMT>(v[j], v[j + 1]), pack_half2<FMT>(v[j + 2], 0.f));
          } else {
            *reinterpret_cast<float4*>(row) = make_float4(v[j], v[j + 1], v[j + 2], 0.f);
          }
        }
      };
      // rows in PAIRS: one proxy fence and one warp barrier per two rows
      uint32_t wa[2], ea[2], wb[2], eb[2], wc[2], ec[2];
      fetch(0, wa[0], ea[0]); fetch(1, wa[1], ea[1]);
      fetch(2, wb[0], eb[0]); fetch(3, wb[1], eb[1]);
      const int nrow = it.rows + 2;
      for (int i = 0; i < nrow; i += 2) {
        fetch(i + 4, wc[0], ec[0]); fetch(i + 5, wc[1], ec[1]);
        const bool two = i + 1 < nrow;
        const int s0 = as;
        const uint32_t p0 = aph;
        if (++as == asl) { as = 0; aph ^= 1; }
        const int s1 = as;
        const uint32_t p1 = aph;
        if (two && ++as == asl) { as = 0; aph ^= 1; }
        mbar_wait(&a_empty[a0 + s0], p0 ^ 1, 0xB00 + s0);
        put(wa[0], ea[0], ring + (size_t)s0 * p.a_slot_bytes);
        if (two) {
          mbar_wait(&a_empty[a0 + s1], p1 ^ 1, 0xB00 + s1);
          put(wa[1], ea[1], ring + (size_t)s1 * p.a_slot_bytes);
        }
        fence_proxy_async();                                      // generic-proxy writes -> visible to the tensor core
        __syncwarp();
        if (lane == 0) { mbar_arrive(&a_full[a0 + s0]); if (two) mbar_arrive(&a_full[a0 + s1]); }
#pragma unroll
        for (int k = 0; k < 2; ++k) { wa[k] = wb[k]; ea[k] = eb[k]; wb[k] = wc[k]; eb[k] = ec[k]; }
      }
    }
  } else if (warp == 0 || (warp == 2 && pipes == 2)) {
    // ================================== input row (A) producer ===================================
    const int pipe = warp >> 1;
    if (elect_one()) {
      const int cps = p.cps, groups = p.cin_chunks / cps;          // a slot holds cps channel chunks of one input row
      const uint32_t slot_tx = (uint32_t)cps * (uint32_t)p.slot_px * rb;
      const int kdl = p.plane ? 1 : p.kd;                          // plane mode: dz is folded, one slot per input plane
      const int a0 = pipe * asl;                                   // this pipeline's slots: [a0, a0 + asl)
      int as = 0;
      uint32_t aph = 0;
      for (int t = blockIdx.x + pipe * gridDim.x; t < p.total_items; t += pipes * gridDim.x) {
        const RowsItem it = rows_decode(p, t);
        for (int i = 0; i < it.rows + 2; ++i)
          for (int dz = 0; dz < kdl; ++dz)
            for (int g = 0; g < groups; ++g) {
              mbar_wait(&a_empty[a0 + as], aph ^ 1, 0xB00 + as);
#ifdef BIU_DBG_KNOBS
              if (g_rows_dbg & 16) { mbar_arrive(&a_full[a0 + as]); if (++as == asl) { as = 0; aph ^= 1; } continue; }
#endif
              mbar_arrive_expect_tx(&a_full[a0 + as], slot_tx);
              for (int c = 0; c < cps; ++c)
                asm volatile(
                    "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, "
                    "%5, %6, %7}], [%2];" ::"r"(a_base + (a0 + as) * p.a_slot_bytes + c * p.a_chunk_bytes),
                    "l"(reinterpret_cast<uint64_t>(&tmA)), "r"(smem_u32(&a_full[a0 + as])),
                    "r"((p.cin_chunk0 + g * cps + c) * p.ck),
                    "r"(it.x0 - 1), "r"(p.plane ? it.y0 - 1 : it.y0 - 1 + i),
                    "r"(p.plane ? i - 1 : it.z - (p.kd >> 1) + dz), "r"(it.b)
                    : "memory");
              if (++as == asl) { as = 0; aph ^= 1; }
            }
      }
    }
  } else if (warp == 1 || (warp == 3 && pipes == 2)) {
    // ====================================== MMA issuer ======================================
    const int pipe = warp >> 1;
    const uint32_t layout = rb == 128 ? 2u : (rb == 64 ? 4u : 6u);
    const uint32_t fmt = fmt_idesc(FMT);
    const uint32_t idesc3 = make_idesc(fmt, (uint32_t)(3 * p.cp));      // whole folded tile
    const uint32_t idesc2 = make_idesc(fmt, (uint32_t)(2 * p.cp));      // split MMAs where the three slots wrap
    const uint32_t idesc1 = make_idesc(fmt, (uint32_t)p.cp);
    const uint64_t a_desc0 = make_smem_desc(a_base + (uint32_t)(pipe * asl) * p.a_slot_bytes, (p.plane ? 10u : 8u) * rb, layout);
    const uint64_t w_desc0 = make_smem_desc(smem_base, 8u * rb, layout);
    constexpr uint32_t px_step = 2u * KS;              // one pixel = row_bytes / 16
    const uint32_t aslot_step = p.a_slot_bytes >> 4, achunk_step = p.a_chunk_bytes >> 4, wtile_step = p.w_tile_bytes >> 4;
    const uint32_t wrow_step = ((uint32_t)p.cp * rb) >> 4;             // cp weight rows (one dy block) further
    const uint32_t wdx_step = p.cin_chunks * wtile_step;               // next dx tap
    mbar_wait(&w_full, 0, 0xC00);
    tc_fence_after();
#ifdef BIU_DBG_KNOBS
    const bool dbg_nomma = (g_rows_dbg & 4) != 0;
#else
    const bool dbg_nomma = false;
#endif
    // This warp's own instruction stream is what bounds the narrow layers (6 MMAs per row: ~550 cycles of
    // bookkeeping against 504 cycles of tensor work, tools/conv_bench.cu), so the per-row path is kept lean: barrier
    // addresses computed once, ring positions as free-running counters (slot = counter & (slots - 1), parity =
    // next bit), no re-derivation of shared-window addresses per barrier operation.
    uint32_t bar_af, bar_ae, bar_tf, bar_te;
    asm volatile("mov.u32 %0, %1;" : "=r"(bar_af) : "r"(smem_u32(a_full + pipe * asl)));
    asm volatile("mov.u32 %0, %1;" : "=r"(bar_ae) : "r"(smem_u32(a_empty + pipe * asl)));
    asm volatile("mov.u32 %0, %1;" : "=r"(bar_tf) : "r"(smem_u32(t_full + pipe * tsl)));
    asm volatile("mov.u32 %0, %1;" : "=r"(bar_te) : "r"(smem_u32(t_empty + pipe * tsl)));
    auto wait_bar = [&](uint32_t addr, uint32_t parity, uint32_t code) {
      uint32_t ok;
      asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                   : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
      if (ok) return;
      const long long t0 = clock64();
      do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                     : "=r"(ok) : "r"(addr), "r"(parity) : "memory");
        if (!ok && clock64() - t0 > 4000000000LL) {
          atomicExch(&g_device_fault, code);
          __threadfence_system();
          asm volatile("trap;");
        }
      } while (!ok);
    };
    auto commit_bar = [&](uint32_t addr) {
      asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(addr) : "memory");
    };
    const uint32_t t_mask = (uint32_t)tsl - 1u, t_lg = tsl == 32 ? 5u : (tsl == 16 ? 4u : 3u), t_wrap = 2u * (uint32_t)tsl - 1u;
    const int kd = p.plane ? 1 : p.kd, chunks = p.cin_chunks, cps = p.cps;
    const bool plane = p.plane != 0;
    const uint32_t cp = (uint32_t)p.cp;
    const uint32_t tmem_pipe = tmem_base + (uint32_t)(pipe * tsl) * cp;   // this pipeline's slot 0
    int as = 0;
    uint32_t aph = 0;
    uint32_t er = 0;                                   // t ring: next virtual row whose slot has to be empty (zeroed)
    uint32_t fr = 0;                                   // t ring: next virtual row to be completed (slot of input row i)
    auto wait_empty = [&]() {
      wait_bar(bar_te + 8u * (er & t_mask), (er >> t_lg) & 1u, 0xD00);
      er = (er + 1u) & t_wrap;
    };
    for (int t = blockIdx.x + pipe * gridDim.x; t < p.total_items; t += pipes * gridDim.x) {
      const int rblk = plane ? 0 : (t / p.strips) % p.rblocks;
      const int rows = plane ? p.D : min(p.RB, p.H - rblk * p.RB);
      wait_empty();                                    // dummy rows v = 0, 1 of this item
      wait_empty();
      for (int i = 0; i < rows + 2; ++i) {
        wait_empty();                                  // virtual row i + 2 receives its first partial row now
        tc_fence_after();
        // input row i accumulates into the slots of virtual rows i, i+1, i+2 (weights ordered dy = 2, 1, 0)
        const uint32_t s0 = fr & t_mask;
        const int wrap = (int)s0 + 3 - tsl;            // > 0: that many slots continue at slot 0
        const uint32_t tcol = tmem_pipe + s0 * cp;
        for (int dz = 0; dz < kd; ++dz)
         for (int g0 = 0; g0 < chunks; g0 += cps) {      // one A slot = cps channel chunks of the row
          wait_bar(bar_af + 8u * (uint32_t)as, aph, 0xE00 + as);
          tc_fence_after();
          for (int c = 0; c < cps; ++c) {
            const int ch = g0 + c;
            const uint64_t ad0 = a_desc0 + (uint64_t)(as * aslot_step + c * achunk_step);
            const uint64_t wd0 = w_desc0 + (uint64_t)((dz * 3 * chunks + ch) * wtile_step);
            if (plane) {
              // nine in-plane taps out of the slot's 18 x 10 halo tile: pixel-row (dy * 10 + dx) further; N = (2-dz, co)
              if (!dbg_nomma && elect_one()) {
                const uint32_t n_lo = wrap == 1 ? idesc2 : idesc1, n_hi = wrap == 1 ? idesc1 : idesc2;
                const uint32_t w_hi = (uint32_t)(3 - wrap) * wrow_step;
#pragma unroll
                for (int dy = 0; dy < 3; ++dy)
#pragma unroll
                  for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                    for (int k = 0; k < KS; ++k) {
                      const uint64_t ad = ad0 + ((dy * 10 + dx) * px_step + 2 * k);
                      const uint64_t wd = wd0 + ((dy * 3 + dx) * wdx_step + 2 * k);
                      if (wrap <= 0) {
                        tc_mma_imm<FMT, 1>(tcol, ad, wd, idesc3);
                      } else {
                        tc_mma_imm<FMT, 1>(tcol, ad, wd, n_lo);
                        tc_mma_imm<FMT, 1>(tmem_pipe, ad, wd + w_hi, n_hi);
                      }
                    }
              }
            } else if (p.first) {
              if (!dbg_nomma && elect_one()) {                     // dx is the K dimension: one MMA per input row
                if (wrap <= 0) {
                  tc_mma_imm<FMT, 1>(tcol, ad0, wd0, idesc3);
                } else {
                  tc_mma_imm<FMT, 1>(tcol, ad0, wd0, wrap == 1 ? idesc2 : idesc1);
                  tc_mma_imm<FMT, 1>(tmem_pipe, ad0, wd0 + (uint32_t)(3 - wrap) * wrow_step, wrap == 1 ? idesc1 : idesc2);
                }
              }
            } else if (!dbg_nomma && elect_one()) {
              if (wrap <= 0) {
#pragma unroll
                for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                  for (int k = 0; k < KS; ++k)
                    tc_mma_imm<FMT, 1>(tcol, ad0 + (dx * px_step + 2 * k), wd0 + (dx * wdx_step + 2 * k), idesc3);
              } else {
                const uint32_t n_lo = wrap == 1 ? idesc2 : idesc1;        // slots before the wrap
                const uint32_t n_hi = wrap == 1 ? idesc1 : idesc2;        // slots continuing at slot 0
                const uint32_t w_hi = (uint32_t)(3 - wrap) * wrow_step;
#pragma unroll
                for (int dx = 0; dx < 3; ++dx)
#pragma unroll
                  for (int k = 0; k < KS; ++k) {
                    tc_mma_imm<FMT, 1>(tcol, ad0 + (dx * px_step + 2 * k), wd0 + (dx * wdx_step + 2 * k), n_lo);
                    tc_mma_imm<FMT, 1>(tmem_pipe, ad0 + (dx * px_step + 2 * k), wd0 + (w_hi + dx * wdx_step + 2 * k), n_hi);
                  }
              }
            }
          }
          if (elect_one()) commit_bar(bar_ae + 8u * (uint32_t)as);
          if (++as == asl) { as = 0; aph ^= 1; }
        }
        if (elect_one()) commit_bar(bar_tf + 8u * s0);   // virtual row i has all its partial rows
        fr = (fr + 1u) & t_wrap;
      }
      // the two trailing dummy rows are complete as well
      if (elect_one()) { commit_bar(bar_tf + 8u * (fr & t_mask)); commit_bar(bar_tf + 8u * ((fr + 1u) & t_mask)); }
      fr = (fr + 2u) & t_wrap;
    }
  } else if (warp >= 4) {
    // ======================================= epilogue =======================================
#define BIU_REPI(CP, MODE, POOL) \
    rows_epilogue<FMT, CP, MODE, POOL>(p, tmem_base, t_full, t_empty, s_scale, s_shift, s_headw, stage, warp, lane)
    if (p.cp == 64) {                                  // plan_rows: 2-byte formats, 2D, EPI_CONV only
      if (ESZ == 2) {
#define BIU_REPI64(POOL, SBW) \
        rows_epilogue<FMT, 64, EPI_CONV, POOL, SBW>(p, tmem_base, t_full, t_empty, s_scale, s_shift, s_headw, stage, warp, lane)
        if (p.stage_px == 32) { if (p.pool_out != nullptr) BIU_REPI64(true, 32); else BIU_REPI64(false, 32); }
        else { if (p.pool_out != nullptr) BIU_REPI64(true, 64); else BIU_REPI64(false, 64); }
#undef BIU_REPI64
      }
    } else if (p.cp == 32) {
      if (p.mode == EPI_HEAD) BIU_REPI(32, EPI_HEAD, false);
      else if (p.pool_out != nullptr) BIU_REPI(32, EPI_CONV, true);
      else BIU_REPI(32, EPI_CONV, false);
    } else {
      if (p.mode == EPI_HEAD) BIU_REPI(16, EPI_HEAD, false);
      else if (p.pool_out != nullptr) BIU_REPI(16, EPI_CONV, true);
      else BIU_REPI(16, EPI_CONV, false);
    }
#undef BIU_REPI
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, 512);
}

#define BIU_ROWS_LAUNCH(E, K)                                                                                     \
  do {                                                                                                             \
    static int max_set = 0;                                                                                        \
    if (smem > max_set) {                                                                                          \
      BIU_CHECK_CUDA(cudaFuncSetAttribute(conv_rows_kernel<E, K>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                          smem));                                                                  \
      max_set = smem;                                                                                              \
    }                                                                                                              \
    conv_rows_kernel<E, K><<<grid, kRowsThreads, smem, stream>>>(tmA, tmW, p);                                     \
  } while (0)
// Host-side dispatch over the k-steps per chunk of one element format.
template <int FMT>
int rows_dispatch(const CUtensorMap& tmA, const CUtensorMap& tmW, const ConvRowsParams& p, int grid, int smem,
                  cudaStream_t stream) {
  const int ks = p.row_bytes / 32;
  if (ks == 4) BIU_ROWS_LAUNCH(FMT, 4); else if (ks == 2) BIU_ROWS_LAUNCH(FMT, 2); else BIU_ROWS_LAUNCH(FMT, 1);
  return 0;
}

// Each element format is instantiated in a translation unit of its own (conv_rows_bf16.cu / _f16.cu / _tf32.cu:
// BIU_ROWS_INSTANCES(, FMT)), so that they compile in parallel; every other unit only declares them.
#define BIU_ROWS_INSTANCES(EXTERN, E)                                                                                \
  EXTERN template int rows_dispatch<E>(const CUtensorMap&, const CUtensorMap&, const ConvRowsParams&, int, int,      \
                                       cudaStream_t);
BIU_ROWS_INSTANCES(extern, FMT_BF16)
BIU_ROWS_INSTANCES(extern, FMT_F16)
BIU_ROWS_INSTANCES(extern, FMT_TF32)

}  // namespace biu
