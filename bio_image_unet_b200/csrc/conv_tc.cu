// Host-side launcher for the tcgen05 implicit-GEMM convolution: builds the TMA tensor maps for the
// activation tensor and the packed weights, picks the pixel box / pipeline depth, launches.
#include "conv_tc.cuh"
#include "conv_halo.cuh"
#include "conv_rows.cuh"
#include "launch.h"
#include <cstdlib>

#include <cudaTypedefs.h>
#include <mutex>

namespace biu {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}
static int pow2_ceil(int v) { return 1 << ilog2(v); }

// Choose a pixel box of exactly 128 pixels: grow along w, then h, then d, then batch.
void choose_box(int W, int H, int D, int B, int* lbw, int* lbh, int* lbd, int* lbb) {
  int rem = 7;
  int lw = ilog2(pow2_ceil(W)); if (lw > rem) lw = rem; rem -= lw;
  // keep the box at most 32 wide when there are rows to stack: better halo locality in L2
  if (lw > 5 && H > 1) { rem += lw - 5; lw = 5; }
  int lh = ilog2(pow2_ceil(H)); if (lh > rem) lh = rem; rem -= lh;
  int ld = ilog2(pow2_ceil(D)); if (ld > rem) ld = rem; rem -= ld;
  int lb = rem;  // whatever is left goes to the batch dim (OOB images are zero-filled and masked)
  *lbw = lw; *lbh = lh; *lbd = ld; *lbb = lb;
}

static CUtensorMapDataType tma_dtype(int fmt) {
  return fmt == FMT_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                         : (fmt == FMT_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32);
}

static int encode_act_map(CUtensorMap* tm, const void* base, int fmt, int C, int W, int H, int D, int B, int ctot,
                          int ck, int bw, int bh, int bd, int bb) {
  EncodeTiledFn enc = get_encode_fn();
  const int esz = fmt_esz(fmt);
  BIU_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  cuuint64_t strides[4] = {(cuuint64_t)ctot * esz, (cuuint64_t)W * ctot * esz, (cuuint64_t)H * W * ctot * esz,
                           (cuuint64_t)D * H * W * ctot * esz};
  cuuint32_t box[5] = {(cuuint32_t)ck, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bd, (cuuint32_t)bb};
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const int rb = ck * esz;
  CUtensorMapSwizzle sw = rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                    : (rb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = enc(tm, tma_dtype(fmt), 5,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BIU_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(activations) failed with %d (C=%d W=%d H=%d D=%d B=%d ctot=%d ck=%d)",
              (int)r, C, W, H, D, B, ctot, ck);
  return 0;
}

static int encode_wgt_map(CUtensorMap* tm, const void* base, int fmt, int cin, int ntotal, int taps, int ck,
                          int n_blk) {
  EncodeTiledFn enc = get_encode_fn();
  const int esz = fmt_esz(fmt);
  BIU_REQUIRE(enc != nullptr, "cuTensorMapEncodeTiled entry point not available");
  cuuint64_t dims[3] = {(cuuint64_t)cin, (cuuint64_t)ntotal, (cuuint64_t)taps};
  cuuint64_t strides[2] = {(cuuint64_t)cin * esz, (cuuint64_t)ntotal * cin * esz};
  cuuint32_t box[3] = {(cuuint32_t)ck, (cuuint32_t)n_blk, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  const int rb = ck * esz;
  CUtensorMapSwizzle sw = rb == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                    : (rb == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  CUresult r = enc(tm, tma_dtype(fmt), 3,
                   const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                   CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  BIU_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(weights) failed with %d (cin=%d n=%d taps=%d ck=%d nblk=%d)",
              (int)r, cin, ntotal, taps, ck, n_blk);
  return 0;
}

int pick_ck(int cin, int fmt) {
  const int esz = fmt_esz(fmt);
  const int cands[3] = {128 / esz, 64 / esz, 32 / esz};
  for (int i = 0; i < 3; ++i)
    if (cin % cands[i] == 0) return cands[i];
  return 0;
}

bool conv_tc_supported(const ConvTcArgs& a) {
  if (a.fmt != FMT_BF16 && a.fmt != FMT_F16 && a.fmt != FMT_TF32) return false;
  const int vec = 16 / fmt_esz(a.fmt);
  if (pick_ck(a.cin, a.fmt) == 0) return false;
  if (a.n_total % 16 != 0) return false;
  if (a.in_ctot % vec != 0 || a.in_coff % vec != 0) return false;
  if (a.mode != EPI_HEAD && (a.out_ctot % vec != 0 || a.out_coff % vec != 0)) return false;
  if (a.mode == EPI_UP && a.up_cout % 16 != 0) return false;
  if (a.mode == EPI_HEAD && (a.n_total > 256 || a.head_n > kMaxHead)) return false;
  return true;
}

// ---------------------------------------------------------------------------------------------------------------
// Halo-tile kernel (conv_halo.cuh): eligibility, tiling choice and launch
// ---------------------------------------------------------------------------------------------------------------
static bool halo_disabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("BIU_CONV_V1"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

#ifdef BIU_DBG_KNOBS
int g_halo_dbg = 0;
int g_halo_force_mt = 0;
int g_halo_force_ck = 0;
#endif

static int sm_count_cached() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

struct HaloPlan { int mt, a_bufs, b_stages, ck, b_resident, stage_bytes, cta2; uint32_t a_buf_bytes, b_stage_bytes; int smem; bool ok; };

// CTA pairs (tcgen05.mma.cta_group::2, conv_halo.cuh): -1 = from the environment (BIU_HALO_NO_CTA2=1 disables)
static int g_halo_cta2 = -1;
void conv_halo_set_cta2(int on) { g_halo_cta2 = on ? 1 : 0; }
static bool halo_cta2_enabled() {
  if (g_halo_cta2 < 0) { const char* e = getenv("BIU_HALO_NO_CTA2"); g_halo_cta2 = (e && e[0] == '1') ? 0 : 1; }
  return g_halo_cta2 == 1;
}

// can the halo kernel take this layer? (3x3(x3) blocks, and transposed convolutions as a 1-tap GEMM)
static bool halo_shape_ok(const ConvTcArgs& a) {
  if (halo_disabled()) return false;
  const bool one = a.kw == 1 && a.kh == 1 && a.kd == 1;      // transposed convolution / 1x1 gate as a plain GEMM
  const bool three = a.kw == 3 && a.kh == 3 && (a.kd == 1 || a.kd == 3);
  if (a.mode == EPI_UP ? !one : !(one || three)) return false;
  if (a.H < 16 || a.W < 8) return false;                 // tiny planes: the per-tap kernel packs the batch instead
  return true;
}

static HaloPlan plan_halo(const ConvTcArgs& a, int n_blk, bool cta2 = false) {
  HaloPlan pl{};
  pl.ok = false;
  if (!halo_shape_ok(a) || n_blk > 256) return pl;
  const int esz = fmt_esz(a.fmt);
  if (cta2 && (n_blk % 32 != 0)) return pl;                // every CTA of a pair stages n_blk / 2 weight rows
  const int halo = a.kw == 3 ? 1 : 0;
  const int rows = 16 + 2 * halo;
  const int taps = halo ? 9 * a.kd : 1;
  // transposed-store staging of the epilogue: 32-channel chunks, conv / transposed conv into one pixel per thread
  const int stage_bytes = (n_blk % 32 == 0 && a.mode != EPI_HEAD && a.out != nullptr &&
                           (a.mode != EPI_UP || a.up_cout % 32 == 0)) ? 8 * 1024 * esz : 0;
  const int extra = (2 * a.n_total + (a.mode == EPI_HEAD ? a.head_n * n_blk : 0)) * 4 + 64 + stage_bytes;   // scale/shift/head
  const int budget = 225 * 1024 - extra;
  const int ck0 = pick_ck(a.cin, a.fmt);
  int mt_max = 256 / n_blk;                                // two accumulator stages of mt * n_blk TMEM columns
  if (mt_max > 8) mt_max = 8;
  const int w8 = (a.W + 7) / 8;
  if (mt_max > w8) mt_max = w8;
#ifdef BIU_DBG_KNOBS
  if (g_halo_force_mt > 0 && mt_max > g_halo_force_mt) mt_max = g_halo_force_mt;
#endif
  while (mt_max & (mt_max - 1)) --mt_max;                  // the kernel is instantiated for mt = 1, 2, 4, 8
  // Preference: two A buffers (load of tile i+1 overlaps the MMAs of tile i), then wide tiles (more MMAs share a
  // weight tile and the halo overhead shrinks), then wide channel chunks.
  for (int abufs = 2; abufs >= 1; --abufs)
    for (int mt = mt_max; mt >= 1; mt >>= 1) {
      if (abufs == 2 && 2 * mt < mt_max) break;            // do not shrink tiles below half for the 2nd buffer
      for (int ck = ck0; ck >= 32 / esz; ck >>= 1) {
        if (a.cin % ck) continue;
#ifdef BIU_DBG_KNOBS
        if (g_halo_force_ck > 0 && ck != g_halo_force_ck) continue;
#endif
        const int rb = ck * esz;
        const int chunks = a.cin / ck;
        const uint32_t tile = ((uint32_t)(a.kd * rows * (8 * mt + 2 * halo) * rb) + 1023u) & ~1023u;
        const uint32_t bst = ((uint32_t)((cta2 ? n_blk / 2 : n_blk) * rb) + 1023u) & ~1023u;
        int stages = (budget - (int)(abufs * tile) - 2048) / (int)bst;
        if (stages > kMaxBStages) stages = kMaxBStages;
        const bool resident = stages >= taps * chunks && a.n_total == n_blk;
        if (stages > taps * chunks) stages = taps * chunks;
        if (stages >= (abufs == 2 ? 3 : 2) || stages == taps * chunks) {
          pl.mt = mt; pl.a_bufs = abufs; pl.b_stages = stages; pl.ck = ck; pl.b_resident = resident ? 1 : 0;
          pl.stage_bytes = stage_bytes; pl.cta2 = cta2 ? 1 : 0;
          pl.a_buf_bytes = tile; pl.b_stage_bytes = bst;
          pl.smem = (int)(abufs * tile + stages * bst) + 1024 + extra;
          pl.ok = true;
          return pl;
        }
      }
    }
  return pl;
}

static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// CTA pairs pay off where a single CTA cannot fetch the weight tile fast enough (N >= 64 columns per MMA: an MMA of N
// columns and K = 16 reads 4096 + 32 N operand bytes at ~85 B/clk for N / 2 cycles of math; a pair halves the weight
// part). Tiles t, t + 1 of a pair must share their weight block (even tile count per block), and the whole grid of pairs
// has to be resident at once (persistent kernel with a static tile stride).
static bool halo_try_cta2(const ConvTcArgs& a, int n_blk, HaloPlan* out, int* pairs_out) {
  if (!halo_cta2_enabled() || n_blk < (a.kd == 3 ? 32 : 64)) return false;   // 27-tap blocks: worth it from N = 32
  if (a.mode == EPI_UP) return false;                     // transposed convolutions are bound by their stores: measured slower in pairs
  HaloPlan pl = plan_halo(a, n_blk, true);
  if (!pl.ok) return false;
  const long long per_block = (long long)ceil_div(a.W, 8 * pl.mt) * ceil_div(a.H, 16) * a.D * a.B;
  if (per_block < 2 || (per_block & 1)) return false;
  static int cache[3][3][4];                               // [format][ks index][mt index] -> pairs + 1 for the largest smem seen
  static int cache_smem[3][3][4];
  const int ks = pl.ck * fmt_esz(a.fmt) / 32, ki = ks == 4 ? 2 : (ks == 2 ? 1 : 0), mi = pl.mt == 8 ? 3 : (pl.mt == 4 ? 2 : (pl.mt == 2 ? 1 : 0));
  const int ei = a.fmt - FMT_BF16;                         // FMT_BF16 / FMT_F16 / FMT_TF32 -> 0 / 1 / 2
  if (cache[ei][ki][mi] == 0 || cache_smem[ei][ki][mi] < pl.smem) {
    const int n =
        with_elem_type(a.fmt, [&](auto tag) { return halo_max_pairs<decltype(tag)::fmt>(ks, pl.mt, pl.smem); });
    cache[ei][ki][mi] = n + 1;
    cache_smem[ei][ki][mi] = pl.smem;
  }
  const int pairs = cache[ei][ki][mi] - 1;
  if (pairs < 1) return false;
  *out = pl;
  *pairs_out = pairs;
  return true;
}

static int launch_conv_halo(const ConvTcArgs& a, int n_blk, const HaloPlan& pl, cudaStream_t stream, int max_pairs = 0) {
  ConvHaloParams p;
  memset(&p, 0, sizeof(p));
  p.W = a.W; p.H = a.H; p.D = a.D; p.B = a.B;
  p.mt = pl.mt;
  p.tiles_x = ceil_div(a.W, 8 * pl.mt);
  p.tiles_y = ceil_div(a.H, 16);
  p.n_blocks = a.n_total / n_blk;
  p.total_tiles = p.tiles_x * p.tiles_y * a.D * a.B * p.n_blocks;
  p.nblk_inner = (p.n_blocks > 1 && !pl.b_resident && !pl.cta2) ? 1 : 0;
  p.kd = a.kd;
  p.halo = a.kw == 3 ? 1 : 0;
  p.ck = pl.ck; p.cin_chunks = a.cin / pl.ck; p.row_bytes = pl.ck * fmt_esz(a.fmt);
  p.n_blk = n_blk; p.n_total = a.n_total;
  p.a_bufs = pl.a_bufs; p.b_stages = pl.b_stages; p.a_buf_bytes = pl.a_buf_bytes; p.b_stage_bytes = pl.b_stage_bytes;
  p.b_resident = pl.b_resident;
  p.cta2 = pl.cta2;
  p.stage_bytes = pl.stage_bytes;
  p.up_cout = a.up_cout; p.up_dims = a.up_dims;
  p.pool_out = a.pool_out; p.pool_ctot = a.pool_ctot; p.pool_coff = a.pool_coff;
  p.mode = a.mode; p.slope = a.slope; p.scale = a.scale; p.shift = a.shift;
  p.out = a.out; p.out_ctot = a.out_ctot; p.out_coff = a.out_coff;
  p.head_n = a.head_n; p.head_w = a.head_w; p.head_b = a.head_b;
  for (int i = 0; i < kMaxHead; ++i) p.head_act[i] = a.head_act[i];
  p.out_val = a.out_val; p.out_u8 = a.out_u8;
#ifdef BIU_DBG_KNOBS
  p.dbg = g_halo_dbg;
#endif

  CUtensorMap tmA, tmB;
  const char* in_base = reinterpret_cast<const char*>(a.in) + (size_t)a.in_coff * fmt_esz(a.fmt);
  if (int rc = encode_act_map(&tmA, in_base, a.fmt, a.cin, a.W, a.H, a.D, a.B, a.in_ctot, pl.ck, 8 * pl.mt + 2 * p.halo, 2, 1, 1))
    return rc;
  if (int rc = encode_wgt_map(&tmB, a.wgt, a.fmt, a.cin, a.n_total, p.halo ? 9 * a.kd : 1, pl.ck, pl.cta2 ? n_blk / 2 : n_blk))
    return rc;
  int grid = p.total_tiles < sm_count() ? p.total_tiles : sm_count();
  if (pl.cta2) {                                           // whole pairs, all of them resident at once
    int pairs = sm_count() / 2;
    if (max_pairs > 0 && pairs > max_pairs) pairs = max_pairs;
    if (pairs > p.total_tiles / 2) pairs = p.total_tiles / 2;
    grid = 2 * pairs;
  }
  BIU_REQUIRE(pl.mt == 1 || pl.mt == 2 || pl.mt == 4 || pl.mt == 8, "halo kernel: mt must be 1, 2, 4 or 8 (got %d)", pl.mt);
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        return halo_dispatch<decltype(tag)::fmt>(tmA, tmB, p, grid, pl.smem, stream);
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Row-streaming folded-tap kernel (conv_rows.cuh): eligibility, plan and launch
// ---------------------------------------------------------------------------------------------------------------
static int g_rows_enabled = -1;     // -1: from the environment (BIU_CONV_NOROWS=1 disables), else 0 / 1
static int g_rows_force_dual = 0;   // test hook (biu_set_rows_kernel(2)): two pipelines even when there are few work items
void conv_rows_set_enabled(int on) { g_rows_enabled = on ? 1 : 0; g_rows_force_dual = on == 2 ? 1 : 0; }
static bool rows_disabled() {
  if (g_rows_enabled < 0) { const char* e = getenv("BIU_CONV_NOROWS"); g_rows_enabled = (e && e[0] == '1') ? 0 : 1; }
  return g_rows_enabled == 0;
}

struct RowsPlan { int ck, cps, stage_px, a_slots, t_slots, RB, smem, plane; uint32_t a_slot_bytes, a_chunk_bytes, w_tile_bytes; bool ok; };

static bool rows_single_pipe() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("BIU_ROWS_SINGLE_PIPE"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

static bool rows_no_wide() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("BIU_ROWS_NO_WIDE"); v = (e && e[0] == '1') ? 1 : 0; }
  return v == 1;
}

static RowsPlan plan_rows(const ConvTcArgs& a) {
  RowsPlan pl{};
  pl.ok = false;
  if (rows_disabled() || halo_disabled() || a.wgt_fold == nullptr) return pl;
  if (a.mode != EPI_CONV && a.mode != EPI_HEAD) return pl;
  if (a.kw != 3 || a.kh != 3 || (a.kd != 1 && a.kd != 3)) return pl;
  // N of the folded MMA = 3 * Cout = 48 or 96; 192 (Cout = 64) for 2D bf16 / fp16 blocks: 8 TMEM slots, one pipeline
  const int esz = fmt_esz(a.fmt);
  const bool wide = a.n_total == 64 && esz == 2 && a.kd == 1 && a.mode == EPI_CONV && !rows_no_wide();
  if (a.n_total != 16 && a.n_total != 32 && !wide) return pl;
  if (a.W < 128) return pl;                                  // one MMA tile = 128 consecutive pixels of a row
  if (a.mode == EPI_HEAD && a.out != nullptr) return pl;
  // fused max-pool: every plane is pooled in (y, x); 3D callers reduce the z pairs afterwards (conv_tc_can_fuse_pool_xy)
  if (a.pool_out != nullptr && ((a.H & 1) || (a.W & 1) || (a.kd == 3 && a.n_total > 32))) return pl;
  if (a.pool_out != nullptr && a.pool_3d) return pl;        // z pairs: plane mode only
  const int ck = pick_ck(a.cin, a.fmt);
  if (ck == 0) return pl;
  const int rb = ck * esz, chunks = a.cin / ck, nfold = 3 * a.n_total;
  pl.ck = ck;
  pl.w_tile_bytes = ((uint32_t)(nfold * rb) + 1023u) & ~1023u;
  pl.a_chunk_bytes = ((uint32_t)(kRowsPx * rb) + 1023u) & ~1023u;
  pl.cps = chunks;
  pl.a_slot_bytes = (uint32_t)chunks * pl.a_chunk_bytes;
  const int px_bytes = a.n_total * esz;
  int stage_px = px_bytes < 64 ? px_bytes : 64;                                          // conv_rows.cuh: SB
  auto tail_of = [&](int spx) { return (2 * a.n_total + kMaxHead * a.n_total) * 4 + 16 * 32 * spx + 64; };   // scale/shift/heads + staging tiles
  const int wbytes = (int)(a.kd * 3 * chunks * pl.w_tile_bytes);
  int tail = tail_of(stage_px);
  int budget = 225 * 1024 - tail - 1024 - wbytes;
  int slots = budget / (int)pl.a_slot_bytes;
  if (slots < 2 * a.kd + 1 && chunks > 1) {
    // a whole input row (all channel chunks) per slot does not leave enough slots: one chunk per slot, and for the
    // 64-channel blocks half-size staging tiles
    pl.cps = 1;
    pl.a_slot_bytes = pl.a_chunk_bytes;
    if (a.n_total == 64) { stage_px = 32; tail = tail_of(stage_px); budget = 225 * 1024 - tail - 1024 - wbytes; }
    slots = budget / (int)pl.a_slot_bytes;
    if (slots < 3 * a.kd) return pl;
  }
  pl.stage_px = stage_px;
  if (slots > kRowsMaxASlots) slots = kRowsMaxASlots;
  if (slots < 2 * a.kd + 1) return pl;                       // weights + a few rows in flight must fit
  pl.a_slots = slots;
  pl.t_slots = 512 / a.n_total;                             // one TMEM slot of Cout columns per output row
  pl.smem = (int)(a.kd * 3 * chunks * pl.w_tile_bytes + slots * pl.a_slot_bytes) + tail + 1024;
  // rows per work item: as tall as possible (2 halo rows per block) while every SM still gets several items
  const long long per_rb1 = (long long)((a.W + 127) / 128) * a.D * a.B;
  pl.RB = 16;
  for (int rbk : {64, 32}) {
    if (per_rb1 * ((a.H + rbk - 1) / rbk) >= 4LL * sm_count_cached()) { pl.RB = rbk; break; }
  }
  pl.ok = true;
  return pl;
}

static int launch_conv_rows(const ConvTcArgs& a, const RowsPlan& pl, cudaStream_t stream, int chunk0 = 0, int nchunks = 0,
                            int acc_mode = 0) {
  ConvRowsParams p;
  memset(&p, 0, sizeof(p));
  p.W = a.W; p.H = a.H; p.D = a.D; p.B = a.B;
  p.strips = (a.W + 127) / 128; p.RB = pl.RB; p.rblocks = (a.H + pl.RB - 1) / pl.RB;
  p.total_items = p.strips * p.rblocks * a.D * a.B;
  p.plane = pl.plane; p.slot_px = pl.plane ? 180 : kRowsPx;
  if (pl.plane) {
    p.tiles_x = (a.W + 7) / 8; p.tiles_y = (a.H + 15) / 16;
    p.strips = 1; p.rblocks = 1;
    p.total_items = p.tiles_x * p.tiles_y * a.B;
  }
  p.kd = a.kd; p.w_taps = a.kd * 3;
  p.ck = pl.ck; p.cin_chunks = nchunks > 0 ? nchunks : a.cin / pl.ck; p.row_bytes = pl.ck * fmt_esz(a.fmt);
  p.cin_chunk0 = chunk0; p.acc_mode = acc_mode; p.acc_scratch = reinterpret_cast<float*>(a.acc_scratch);
  p.cp = a.n_total;
  p.a_slots = pl.a_slots; p.a_slot_bytes = pl.a_slot_bytes; p.a_chunk_bytes = pl.a_chunk_bytes; p.cps = pl.cps; p.stage_px = pl.stage_px;
  // two pipelines per CTA when the A ring is deep enough to be halved and there is work for both
  static int min_slots = -1;
  if (min_slots < 0) { const char* e = getenv("BIU_ROWS_PIPE_MIN_SLOTS"); min_slots = e ? atoi(e) : 8; }
  p.pipes = (pl.a_slots >= min_slots && (p.total_items >= 2 * sm_count_cached() || g_rows_force_dual) && !rows_single_pipe() &&
             a.n_total <= 32) ? 2 : 1;
  if (p.pipes == 2) p.a_slots &= ~1;
  p.w_tile_bytes = pl.w_tile_bytes; p.t_slots = pl.t_slots;
  p.mode = a.mode; p.slope = a.slope; p.scale = a.scale; p.shift = a.shift;
  p.out = a.out; p.out_ctot = a.out_ctot; p.out_coff = a.out_coff;
  p.pool_out = a.pool_out; p.pool_ctot = a.pool_ctot; p.pool_coff = a.pool_coff;
  p.head_n = a.head_n; p.head_w = a.head_w; p.head_b = a.head_b;
  for (int i = 0; i < kMaxHead; ++i) p.head_act[i] = a.head_act[i];
  p.out_val = a.out_val; p.out_u8 = a.out_u8;
  CUtensorMap tmA, tmW;
  const char* in_base = reinterpret_cast<const char*>(a.in) + (size_t)a.in_coff * fmt_esz(a.fmt);
  if (int rc = pl.plane ? encode_act_map(&tmA, in_base, a.fmt, a.cin, a.W, a.H, a.D, a.B, a.in_ctot, pl.ck, 10, 18, 1, 1)
                        : encode_act_map(&tmA, in_base, a.fmt, a.cin, a.W, a.H, a.D, a.B, a.in_ctot, pl.ck, kRowsPx, 1, 1, 1))
    return rc;
  if (int rc = encode_wgt_map(&tmW, pl.plane ? a.wgt_fold_z : a.wgt_fold, a.fmt, a.cin, 3 * a.n_total, a.kd * 3, pl.ck, 3 * a.n_total))
    return rc;
  const int grid = p.total_items < sm_count_cached() ? p.total_items : sm_count_cached();
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        return rows_dispatch<decltype(tag)::fmt>(tmA, tmW, p, grid, pl.smem, stream);
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------------
// First block of the 2D nets on the row kernel's first mode (conv_rows.cuh): the producer warps build the 32-byte A rows
// {in[x-1], in[x], in[x+1], 0...} from the uint8 tile, one MMA of N = 3 * Cout per input row.
// ---------------------------------------------------------------------------------------------------------------------
static bool first_rows_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("BIU_FIRST_NO_ROWS"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}
bool conv_first_rows_supported(const FirstRowsArgs& a) {
  if (!first_rows_enabled() || rows_disabled() || halo_disabled()) return false;
  if (a.wgt == nullptr || (a.n_total != 16 && a.n_total != 32) || (a.fmt != FMT_BF16 && a.fmt != FMT_F16 && a.fmt != FMT_TF32))
    return false;
  return a.W >= 128 && a.H >= 1 && a.out_ctot % 8 == 0 && a.out_coff % 8 == 0;
}
int launch_conv_first_rows(const FirstRowsArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(conv_first_rows_supported(a), "first block on the row kernel: unsupported configuration (n=%d W=%d)", a.n_total, a.W);
  ConvRowsParams p;
  memset(&p, 0, sizeof(p));
  const int rb = 32, nfold = 3 * a.n_total;
  p.W = a.W; p.H = a.H; p.D = 1; p.B = a.B;
  p.strips = (a.W + 127) / 128;
  const long long per_rb1 = (long long)p.strips * a.B;
  p.RB = 16;
  for (int rbk : {64, 32}) {
    if (per_rb1 * ((a.H + rbk - 1) / rbk) >= 4LL * sm_count_cached()) { p.RB = rbk; break; }
  }
  p.rblocks = (a.H + p.RB - 1) / p.RB;
  p.total_items = p.strips * p.rblocks * a.B;
  p.kd = 1; p.slot_px = 128; p.first = 1; p.first_in = a.in; p.w_taps = 1;
  p.ck = rb / fmt_esz(a.fmt); p.cin_chunks = 1; p.row_bytes = rb; p.cps = 1;
  p.cp = a.n_total;
  p.a_chunk_bytes = 128 * rb; p.a_slot_bytes = p.a_chunk_bytes;
  p.w_tile_bytes = ((uint32_t)(nfold * rb) + 1023u) & ~1023u;
  const int px_bytes = a.n_total * fmt_esz(a.fmt);
  p.stage_px = px_bytes < 64 ? px_bytes : 64;
  const int tail = (2 * a.n_total + kMaxHead * a.n_total) * 4 + 16 * 32 * p.stage_px + 64;
  p.a_slots = kRowsMaxASlots;
  p.t_slots = 512 / a.n_total;
  p.pipes = (p.total_items >= 2 * sm_count_cached() && !rows_single_pipe()) ? 2 : 1;
  const int smem = (int)p.w_tile_bytes + p.a_slots * (int)p.a_slot_bytes + tail + 1024;
  p.mode = EPI_CONV; p.slope = a.slope; p.scale = a.scale; p.shift = a.shift;
  p.out = a.out; p.out_ctot = a.out_ctot; p.out_coff = a.out_coff;
  CUtensorMap tmW;
  if (int rc = encode_wgt_map(&tmW, a.wgt, a.fmt, p.ck, nfold, 1, p.ck, nfold)) return rc;
  const int grid = p.total_items < sm_count_cached() ? p.total_items : sm_count_cached();
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {      // no activation map: the rows are built in the kernel
        return rows_dispatch<decltype(tag)::fmt>(tmW, tmW, p, grid, smem, stream);
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

static int choose_n_blk(const ConvTcArgs& a) {
  // N per CTA: whole N when it fits one accumulator, otherwise the largest divisor <= 256
  int n_blk = a.n_total;
  if (n_blk > 256) {
    n_blk = 256;
    while (a.n_total % n_blk != 0) n_blk -= 16;
  }
  if (a.mode == EPI_UP && n_blk > a.up_cout && n_blk % a.up_cout != 0) n_blk = a.up_cout;
  return n_blk;
}

// Plane mode of the row kernel (conv_rows.cuh): 3x3x3 blocks with Cout <= 32 on planes narrower than 128 px (the
// level-1 layers of the 3D nets). The M tile is a 16 x 8 pixel tile, the dz taps are folded into N and the planes of
// the tile stream through the TMEM slot ring: N = 3 * Cout per MMA instead of the halo-tile kernel's N = Cout.
static bool rows_plane_enabled() {
  static int v = -1;
  if (v < 0) { const char* e = getenv("BIU_ROWS_NO_PLANE"); v = (e && e[0] == '1') ? 0 : 1; }
  return v == 1;
}
// chunks_limit > 0: plan for a launch that covers only that many channel chunks of the block (K split)
static RowsPlan plan_rows_plane(const ConvTcArgs& a, int chunks_limit = 0) {
  RowsPlan pl{};
  pl.ok = false;
  if (rows_disabled() || halo_disabled() || !rows_plane_enabled() || a.wgt_fold_z == nullptr) return pl;
  if (a.mode != EPI_CONV && a.mode != EPI_HEAD) return pl;
  // fused MaxPool3d(2): the planes of a tile come in pairs (z), the 16 x 8 tile holds whole (y, x) pairs
  if (a.pool_out != nullptr && (!a.pool_3d || a.mode != EPI_CONV || (a.D & 1) || (a.H & 1) || (a.W & 1))) return pl;
  if (a.mode == EPI_CONV ? a.out == nullptr : a.out != nullptr) return pl;      // heads: no feature output
  if (a.kw != 3 || a.kh != 3 || a.kd != 3 || a.D < 2) return pl;
  if (a.n_total != 16 && a.n_total != 32) return pl;
  if (a.W < 8 || a.H < 16) return pl;                        // tiny planes: the halo / per-tap kernels (wide ones try the row mode first)
  const int ck = pick_ck(a.cin, a.fmt);
  if (ck == 0) return pl;
  const int esz = fmt_esz(a.fmt);
  const int rb = ck * esz, chunks = chunks_limit > 0 ? chunks_limit : a.cin / ck, nfold = 3 * a.n_total;
  pl.plane = 1;
  pl.ck = ck;
  pl.w_tile_bytes = ((uint32_t)(nfold * rb) + 1023u) & ~1023u;
  pl.a_chunk_bytes = ((uint32_t)(180 * rb) + 1023u) & ~1023u;      // 18 x 10 halo tile of one plane and channel chunk
  const int px_bytes = a.n_total * esz;
  pl.stage_px = px_bytes < 64 ? px_bytes : 64;
  const int tail = (2 * a.n_total + kMaxHead * a.n_total) * 4 + 16 * 32 * pl.stage_px + 64;
  const int wbytes = (int)(9 * chunks * pl.w_tile_bytes);
  const int budget = 225 * 1024 - tail - 1024 - wbytes;
  pl.cps = chunks;
  pl.a_slot_bytes = (uint32_t)chunks * pl.a_chunk_bytes;
  int slots = budget / (int)pl.a_slot_bytes;
  if (slots < 3 && chunks > 1) {                            // one channel chunk per slot
    pl.cps = 1;
    pl.a_slot_bytes = pl.a_chunk_bytes;
    slots = budget / (int)pl.a_slot_bytes;
  }
  // The nine-tap weights of every channel chunk are resident: with 96 input channels (decode3 of UNet3D) they take 162 KB
  // and leave three single-chunk slots - too few to cover the TMA latency (measured 16.3 ms against 15.7 ms on the
  // halo-tile kernel, which streams its weights), so such blocks stay there.
  if (slots < 6) return pl;
  if (slots > kRowsMaxASlots) slots = kRowsMaxASlots;
  pl.a_slots = slots;
  pl.t_slots = 512 / a.n_total;
  pl.smem = wbytes + slots * (int)pl.a_slot_bytes + tail + 1024;
  pl.RB = a.D;
  pl.ok = true;
  return pl;
}

// 3D blocks both modes can take (planes >= 128 px wide): the plane mode loads every input plane of a tile once instead
// of every row three times (once per dz), needs no halo rows, and pools in (z, y, x). Measured on UNet3D(16) at
// 64 x 128 x 128, ms per 256 patches, row -> plane mode: encode2 + pool 9.4 -> 7.8, decode5 (48 -> 16, 8-slot ring)
// 14.5 -> 12.0, decode6 + head 7.6 -> 5.5; MO-3D full-resolution blocks 1.12 -> 0.76 and 1.98 -> 1.70 per forward.
// Preferred when its ring holds at least BIU_ROWS_PLANE_MIN_SLOTS (default 8) tiles; BIU_ROWS_PLANE_FIRST=0 / 1 forces
// the choice (A/B runs).
static bool rows_plane_preferred(const RowsPlan& pp) {
  static int plane_first = -1;
  if (plane_first < 0) { const char* e = getenv("BIU_ROWS_PLANE_FIRST"); plane_first = e ? (e[0] == '1' ? 1 : 0) : 2; }
  static int min_slots = -1;
  if (min_slots < 0) { const char* e = getenv("BIU_ROWS_PLANE_MIN_SLOTS"); min_slots = e ? atoi(e) : 8; }
  return pp.ok && (plane_first == 1 || (plane_first == 2 && pp.a_slots >= min_slots));
}

bool conv_tc_can_fuse_pool3d(const ConvTcArgs& a) {
  if (!conv_tc_supported(a) || a.mode != EPI_CONV || a.kd != 3 || !a.pool_3d) return false;
  return rows_plane_preferred(plan_rows_plane(a));
}
bool conv_tc_can_fuse_pool_xy(const ConvTcArgs& a) {
  // 3D blocks: only the row kernel pools (plane by plane, in y and x)
  if (!conv_tc_supported(a) || a.mode != EPI_CONV || a.kd != 3 || (a.H & 1) || (a.W & 1) || (a.D & 1)) return false;
  return plan_rows(a).ok;
}
bool conv_tc_can_fuse_pool(const ConvTcArgs& a) {
  if (!conv_tc_supported(a) || a.mode != EPI_CONV || a.kd != 1 || a.D != 1 || (a.H & 1) || (a.W & 1)) return false;
  return plan_rows(a).ok || plan_halo(a, choose_n_blk(a)).ok;
}

int launch_conv_tc(const ConvTcArgs& a, cudaStream_t stream) {
  BIU_REQUIRE(conv_tc_supported(a), "conv_tc: unsupported configuration (cin=%d n=%d fmt=%d mode=%d)", a.cin,
              a.n_total, a.fmt, a.mode);
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  p.W = a.W; p.H = a.H; p.D = a.D; p.B = a.B;
  choose_box(a.W, a.H, a.D, a.B, &p.lbw, &p.lbh, &p.lbd, &p.lbb);
  p.tiles_w = ceil_div(a.W, 1 << p.lbw);
  p.tiles_h = ceil_div(a.H, 1 << p.lbh);
  p.tiles_d = ceil_div(a.D, 1 << p.lbd);
  p.tiles_b = ceil_div(a.B, 1 << p.lbb);
  p.kw = a.kw; p.kh = a.kh; p.kd = a.kd;
  p.ck = pick_ck(a.cin, a.fmt);
  p.cin_chunks = a.cin / p.ck;
  p.row_bytes = p.ck * fmt_esz(a.fmt);
  {
    const RowsPlan pp = plan_rows_plane(a);
    {
      static int dbg = -1;
      if (dbg < 0) { const char* e = getenv("BIU_PLAN_DEBUG"); dbg = (e && e[0] == '1') ? 1 : 0; }
      if (dbg && a.kd == 3) {
        const RowsPlan rp0 = plan_rows(a);
        fprintf(stderr, "[plan] cin=%d n=%d %dx%dx%d B=%d mode=%d pool=%d/%d | rows ok=%d slots=%d cps=%d RB=%d | plane ok=%d slots=%d cps=%d ck=%d\n",
                a.cin, a.n_total, a.D, a.H, a.W, a.B, a.mode, a.pool_out != nullptr, a.pool_3d, rp0.ok, rp0.a_slots, rp0.cps,
                rp0.RB, pp.ok, pp.a_slots, pp.cps, pp.ck);
      }
    }
    if (pp.ok && (a.pool_3d || rows_plane_preferred(pp))) return launch_conv_rows(a, pp, stream);
    const RowsPlan rp = plan_rows(a);
    if (rp.ok) return launch_conv_rows(a, rp, stream);
    if (pp.ok) return launch_conv_rows(a, pp, stream);
    // K split: the nine-tap weights of all channel chunks do not fit beside a usable A ring (96 input channels: 162 KB).
    // Run the block as several launches over groups of chunks; the partial sums travel through an fp32 scratch.
    if (a.acc_scratch != nullptr && a.cin > 0 && a.mode == EPI_CONV) {
      const int ck = pick_ck(a.cin, a.fmt);
      const int chunks = ck ? a.cin / ck : 0;
      const long long need = (long long)a.B * a.D * a.H * a.W * a.n_total * 4;
      int group = 0;
      RowsPlan gp{};
      for (int g = chunks - 1; g >= 1; --g) {
        gp = plan_rows_plane(a, g);
        if (gp.ok) { group = g; break; }
      }
      if (group > 0 && chunks > group && need <= a.acc_scratch_bytes) {
        for (int c0 = 0; c0 < chunks; c0 += group) {
          const int n = chunks - c0 < group ? chunks - c0 : group;
          const bool first = c0 == 0, last = c0 + n >= chunks;
          const RowsPlan lp = n == group ? gp : plan_rows_plane(a, n);
          BIU_REQUIRE(lp.ok, "conv_rows K split: no plan for %d channel chunks", n);
          if (int rc = launch_conv_rows(a, lp, stream, c0, n, first ? 1 : (last ? 2 : 3))) return rc;
        }
        return 0;
      }
    }
  }
  const int n_blk = choose_n_blk(a);
  {
    HaloPlan pl2;
    int pairs = 0;
    if (halo_try_cta2(a, n_blk, &pl2, &pairs)) return launch_conv_halo(a, n_blk, pl2, stream, pairs);
    const HaloPlan pl = plan_halo(a, n_blk);
    if (pl.ok) return launch_conv_halo(a, n_blk, pl, stream);
  }
  BIU_REQUIRE(a.pool_out == nullptr, "conv_tc: the fused max-pool needs the halo-tile kernel (check conv_tc_can_fuse_pool)");
  p.n_blk = n_blk;
  p.mode = a.mode;
  p.slope = a.slope;
  p.scale = a.scale; p.shift = a.shift;
  p.out = a.out; p.out_ctot = a.out_ctot; p.out_coff = a.out_coff;
  p.up_cout = a.up_cout; p.up_dims = a.up_dims;
  p.head_n = a.head_n; p.head_w = a.head_w; p.head_b = a.head_b;
  for (int i = 0; i < kMaxHead; ++i) p.head_act[i] = a.head_act[i];
  p.out_val = a.out_val; p.out_u8 = a.out_u8;

  const int a_bytes = 128 * p.row_bytes;
  const int b_bytes = (n_blk * p.row_bytes + 1023) & ~1023;
  const int stage_bytes = a_bytes + b_bytes;
  const int num_kb = p.cin_chunks * a.kw * a.kh * a.kd;
  int stages = (a.smem_budget > 0 ? a.smem_budget : 96 * 1024) / stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages > num_kb) stages = num_kb;
  if (stages < 2) stages = num_kb < 2 ? 1 : 2;
  p.stages = stages;
  const int smem = stages * stage_bytes + 1024;

  CUtensorMap tmA, tmB;
  const char* in_base = reinterpret_cast<const char*>(a.in) + (size_t)a.in_coff * fmt_esz(a.fmt);
  if (int rc = encode_act_map(&tmA, in_base, a.fmt, a.cin, a.W, a.H, a.D, a.B, a.in_ctot, p.ck, 1 << p.lbw,
                              1 << p.lbh, 1 << p.lbd, 1 << p.lbb))
    return rc;
  if (int rc = encode_wgt_map(&tmB, a.wgt, a.fmt, a.cin, a.n_total, a.kw * a.kh * a.kd, p.ck, n_blk)) return rc;

  dim3 grid(p.tiles_w * p.tiles_h * p.tiles_d * p.tiles_b, a.n_total / n_blk);
  if (int rc = with_elem_type(a.fmt, [&](auto tag) {
        constexpr int FMT = decltype(tag)::fmt;
        static int max_set = 0;
        if (smem > max_set) {
          BIU_CHECK_CUDA(cudaFuncSetAttribute(conv_tc_kernel<FMT>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
          max_set = smem;
        }
        conv_tc_kernel<FMT><<<grid, 192, smem, stream>>>(tmA, tmB, p);
        return 0;
      }))
    return rc;
  BIU_CHECK_CUDA(cudaGetLastError());
  count_launch();
  return 0;
}

int read_device_fault(unsigned int* out) {
  BIU_CHECK_CUDA(cudaMemcpyFromSymbol(out, g_device_fault, sizeof(unsigned int)));
  return 0;
}

}  // namespace biu
