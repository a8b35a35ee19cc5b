// Single-layer timing harness for the tcgen05 convolution kernels (development aid, not part of the product).
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -DBIU_DBG_KNOBS -o tools/conv_bench tools/conv_bench.cu -lcuda
// Usage: conv_bench [tiles]   -- times the cfg-2 Unet(32) layer shapes on `tiles` 512x512 tiles with every debug knob
#include "../bio_image_unet_b200/csrc/conv_tc.cu"
#include "../bio_image_unet_b200/csrc/conv_halo_bf16.cu"
#include "../bio_image_unet_b200/csrc/conv_halo_f16.cu"
#include "../bio_image_unet_b200/csrc/conv_halo_tf32.cu"
#include "../bio_image_unet_b200/csrc/conv_rows_bf16.cu"
#include "../bio_image_unet_b200/csrc/conv_rows_f16.cu"
#include "../bio_image_unet_b200/csrc/conv_rows_tf32.cu"
#include <vector>
#include <cstdarg>
namespace biu {
static char g_err[1024];
void set_error(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof(g_err), fmt, ap); va_end(ap); }
const char* get_error() { return g_err; }
unsigned long long g_launch_count = 0;
}
using namespace biu;

static int g_use_rows = 0;
struct LayerCfg { const char* name; int cin, cout, level; int up; };

static float time_layer(const LayerCfg& L, int tiles, void* in, void* wgt, float* scale, float* shift, void* out, int reps) {
  const int H = 512 >> L.level, W = 512 >> L.level;
  ConvTcArgs a;
  memset(&a, 0, sizeof(a));
  a.fmt = FMT_BF16; a.in = in; a.in_ctot = L.cin; a.in_coff = 0; a.cin = L.cin; a.W = W; a.H = H; a.D = 1; a.B = tiles;
  if (!L.up) {
    a.kw = a.kh = 3; a.kd = 1; a.n_total = L.cout; a.mode = EPI_CONV; a.slope = 0.1f;
    a.out_ctot = L.cout;
  } else {
    a.kw = a.kh = a.kd = 1; a.n_total = 4 * L.cout; a.mode = EPI_UP; a.slope = 1.f; a.up_cout = L.cout; a.up_dims = 2;
    a.out_ctot = 2 * L.cout;
  }
  a.wgt = wgt; a.wgt_fold = (g_use_rows && !L.up) ? wgt : nullptr; a.scale = scale; a.shift = shift; a.out = out; a.out_coff = 0;
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  if (launch_conv_tc(a, 0)) { printf("launch failed: %s\n", get_error()); return -1; }
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { printf("kernel failed: %s\n", cudaGetErrorString(e)); exit(1); }
  cudaEventRecord(e0);
  for (int r = 0; r < reps; ++r) launch_conv_tc(a, 0);
  cudaEventRecord(e1);
  cudaEventSynchronize(e1);
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  return ms / reps;
}

int main(int argc, char** argv) {
  const int tiles = argc > 1 ? atoi(argv[1]) : 48;
  const int reps = argc > 2 ? atoi(argv[2]) : 3;
  const LayerCfg layers[] = {
      {"encode2 32->32 @512", 32, 32, 0, 0},   {"decode7 64->32 @512", 64, 32, 0, 0},
      {"encode4 64->64 @256", 64, 64, 1, 0},   {"decode5 128->64 @256", 128, 64, 1, 0},
      {"encode6 128->128 @128", 128, 128, 2, 0}, {"decode3 256->128 @128", 256, 128, 2, 0},
      {"decode1 512->256 @64", 512, 256, 3, 0}, {"mid2 512->512 @32", 512, 512, 4, 0},
      {"up4 64->32 @256", 64, 32, 1, 1},       {"up3 128->64 @128", 128, 64, 2, 1},
      {"up2 256->128 @64", 256, 128, 3, 1},    {"up1 512->256 @32", 512, 256, 4, 1}};
  const size_t max_act = (size_t)tiles * 512 * 512 * 64 * 2;   // largest activation tensor: 64 ch at full res
  void *in, *out, *wgt; float *scale, *shift;
  cudaMalloc(&in, max_act); cudaMalloc(&out, max_act);
  cudaMalloc(&wgt, (size_t)9 * 512 * 512 * 2);
  cudaMalloc(&scale, 4096 * 4); cudaMalloc(&shift, 4096 * 4);
  {
    std::vector<uint16_t> h(max_act / 2 > (1u << 26) ? (1u << 26) : max_act / 2);
    for (size_t i = 0; i < h.size(); ++i) h[i] = (uint16_t)(0x3c00 + (i * 2654435761u >> 22 & 0x3ff));   // bf16 ~ [0.0078, 0.03]
    for (size_t off = 0; off < max_act; off += h.size() * 2)
      cudaMemcpy((char*)in + off, h.data(), std::min(h.size() * 2, max_act - off), cudaMemcpyHostToDevice);
    std::vector<uint16_t> w((size_t)9 * 512 * 512);
    for (size_t i = 0; i < w.size(); ++i) w[i] = (uint16_t)(0x3c00 + (i * 40503u & 0xff));
    cudaMemcpy(wgt, w.data(), w.size() * 2, cudaMemcpyHostToDevice);
    std::vector<float> s(4096, 1.0f), z(4096, 0.0f);
    cudaMemcpy(scale, s.data(), 4096 * 4, cudaMemcpyHostToDevice);
    cudaMemcpy(shift, z.data(), 4096 * 4, cudaMemcpyHostToDevice);
  }
  const int knobs[] = {0, 64, 8, 8 | 64, 2, 4 | 2, 4 | 2 | 1, 4 | 2 | 32 | 1, 2 | 8, 4 | 2 | 8};
  const char* knob_names[] = {"full", "alignA", "-epi", "-epi+algn", "-mma", "-A-mma", "-A-mma-st", "-A-mma-stma", "-mma-epi", "-A-mma-epi"};
  printf("%-24s", "layer (ms)");
  for (auto k : knob_names) printf("%11s", k);
  printf("%10s%10s\n", "TFLOP/s", "GB/s");
  const bool rows_only = argc > 3 && argv[3][0] == 'r';
  for (const LayerCfg& L : layers) {
    if (rows_only) break;
    printf("%-24s", L.name);
    float full = 0;
    for (size_t k = 0; k < sizeof(knobs) / sizeof(int); ++k) {
      g_halo_dbg = knobs[k];
      float ms = time_layer(L, tiles, in, wgt, scale, shift, out, reps);
      if (k == 0) full = ms;
      printf("%11.3f", ms);
    }
    const double px = (double)tiles * (512 >> L.level) * (512 >> L.level);
    const double fl = 2.0 * px * L.cout * L.cin * (L.up ? 4 : 9);
    const double bytes = px * 2.0 * (L.cin + (L.up ? 4 : 1) * L.cout);
    printf("%10.1f%10.0f\n", fl / full / 1e9, bytes / full / 1e6);
    fflush(stdout);
  }
  if (argc > 3 && !rows_only) {  // mt sweep on the first two layers
    for (int mt : {8, 4, 2, 1}) {
      g_halo_force_mt = mt; g_halo_dbg = 0;
      for (int li : {0, 1, 2, 3, 8, 9})
        printf("mt<=%d %-24s %8.3f ms\n", mt, layers[li].name, time_layer(layers[li], tiles, in, wgt, scale, shift, out, reps));
    }
    g_halo_force_mt = 0;
    for (int ck : {64, 32, 16}) {
      g_halo_force_ck = ck;
      for (int li : {1, 2, 3, 5, 8, 9})
        printf("ck=%d %-24s %8.3f ms\n", ck, layers[li].name, time_layer(layers[li], tiles, in, wgt, scale, shift, out, reps));
    }
    g_halo_force_ck = 0;
  }
  {  // row-streaming kernel on the narrow layers: full / one TMEM load per row / no TMEM loads / no MMA
    g_halo_dbg = 0; g_use_rows = 1;
    for (int li : {0, 1}) {
      printf("rows kernel %-24s", layers[li].name);
      for (int k : {0, 8, 64, 4, 64 | 4, 116}) {
        cudaMemcpyToSymbol(g_rows_dbg, &k, sizeof(int));
        printf("  dbg%d %.3f ms", k, time_layer(layers[li], tiles, in, wgt, scale, shift, out, reps));
      }
      printf("\n");
    }
    int z = 0; cudaMemcpyToSymbol(g_rows_dbg, &z, sizeof(int));
    g_use_rows = 0;
  }
  if (!rows_only) {  // cycle accounting of CTA 0
    const char* slot_names[12] = {"A: wait a_empty", "A: issue TMA", "B: wait b_empty", "MMA: wait acc_empty", "MMA: wait a_full",
                                  "MMA: wait b_full", "MMA: issue+commit", "-", "EPI(w4): wait acc_full", "EPI: tmem wait",
                                  "EPI: whole tile", "EPI: arrive"};
    for (int li : {0, 0, 0, 1, 2, 8}) {
      static int call = 0;
      unsigned long long z[32] = {0}, h[32];
      cudaMemcpyToSymbol(g_halo_prof, z, sizeof(z));
      g_halo_dbg = 256 | (call == 1 ? (4 | 2) : (call == 2 ? (4 | 2 | 1 | 32) : 0)); g_halo_force_mt = 0;
      printf("dbg=%d ", g_halo_dbg);
      ++call;
      float ms = time_layer(layers[li], tiles, in, wgt, scale, shift, out, 1);
      cudaMemcpyFromSymbol(h, g_halo_prof, sizeof(h));
      printf("--- %s: %.3f ms per launch; CTA0 kilo-cycles over 2 launches:\n", layers[li].name, ms);
      for (int i = 0; i < 12; ++i) if (i != 7) printf("    %-24s %10.1f\n", slot_names[i], h[i] / 1e3);
    }
  }
  unsigned int fault = 0;
  read_device_fault(&fault);
  printf("device fault word: %u\n", fault);
  return 0;
}
