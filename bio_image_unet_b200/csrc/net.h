// Network handle behind the C-ABI: holds the reference checkpoint's tensors (by state_dict name), folds
// BatchNorm, packs weights for the tensor-core kernels and runs the layer program of one of the reference's
// model families on a batch of tiles.
#pragma once
#include <cuda_runtime.h>
#include <map>
#include <string>
#include <vector>
#include "launch.h"

namespace biu {

enum NetKind { NET_UNET2D = 0, NET_SIAM2D = 1, NET_UNET3D = 2, NET_MO3D = 3, NET_UNET2D_V0 = 4, NET_ATTUNET2D = 5, NET_MO2D = 6,
               NET_NESTED2D = 7, NET_NESTED2D_3L = 8 };
enum SiamMode { SIAM_CONCAT = 0, SIAM_MAX = 1, SIAM_CONTROL = 2, SIAM_CORR = 3 };

struct HostTensor {
  std::vector<long long> shape;
  std::vector<float> data;
};

struct Segment {       // logical input channels [lstart, lstart+count) live at physical channel pstart
  int lstart, count, pstart;
};

struct ConvLayer {     // one Conv+BN+LeakyReLU block, a transposed conv, or the head
  std::string name;
  std::string conv_key, bn_key;   // state_dict prefixes of the conv and its BatchNorm; empty: '<name>.0' / '<name>.1'
  int cin_log = 0, cout = 0, cin_phys = 0, cout_pad = 0;
  int kd = 1, kh = 1, kw = 1;
  bool is_up = false;
  bool is_gate = false;      // AttentionBlock: 1x1 convs of gate + skip folded into one GEMM, psi as its 1x1 head
  int nq = 1;
  float slope = 0.1f;        // LeakyReLU slope of the block (0 = ReLU: Unet_v0, attention gate)
  float* gate_w = nullptr;   // is_gate: psi weights [cout_pad] and bias [1] (BatchNorm(1) folded)
  float* gate_b = nullptr;
  std::vector<Segment> segs;
  void* w_tc = nullptr;      // packed [tap][n][cin_phys] in the net's format (bf16 / fp16 / tf32)
  void* w_fold = nullptr;    // narrow 3x3 blocks: [dz*3+dx][(2-dy)*cout_pad + co][cin_phys] for the row-streaming kernel
  void* w_fold_z = nullptr;  // narrow 3x3x3 blocks: [dy*3+dx][(2-dz)*cout_pad + co][cin_phys] for its plane mode (dz folded)
  float* w_direct = nullptr; // fp32 [tap or q][cin_phys][cout_pad]
  void* w_first = nullptr;   // first block of the 2D nets (1 input channel): [(2-dy)*cout_pad + co][dx, zeros] bf16 / fp16 x16, tf32 x8
  float* scale_first = nullptr;   // scale / 255 (conv_rows.cuh first mode works on the raw uint8 values)
  float* scale = nullptr;    // [n_total]
  float* shift = nullptr;
};

enum OpKind { OP_FIRST, OP_CONV, OP_CONV_HEAD, OP_UP, OP_POOL, OP_UPNEAREST, OP_MAXJOIN, OP_GATE, OP_MULPSI, OP_XCORR, OP_UPTRILINEAR, OP_UPBILINEAR };

struct Op {
  OpKind kind;
  int layer = -1;            // index into layers
  int src = -1, dst = -1;    // buffer ids (-1: network input / output)
  int src_coff = 0, dst_coff = 0, c = 0;
  int src_img0 = 0, dst_img0 = 0;   // image offsets in units of the plan batch B
  int batch_mul = 1;         // op runs on batch_mul * B images
  int level = 0;
  int pool_mode = 0;
  int src2 = -1;             // OP_MAXJOIN second operand image offset
};

struct Buf {
  std::string name;
  int level = 0, ctot = 0, batch_mul = 1;
  size_t offset = 0;
};

struct Net {
  int kind = 0, dims = 2, nf = 32, in_ch = 1;
  int fmt = 0;                      // ElemFmt (common.cuh) of the activations and tensor-core weights
  int siam_mode = 0, use_interp = 0;
  int levels = 4;
  std::vector<int> head_channels;   // per head
  std::vector<int> head_acts;       // per head
  std::vector<std::string> head_names;
  int head_total = 0;
  std::map<std::string, HostTensor> params;
  bool finalized = false;

  std::vector<ConvLayer> layers;
  std::vector<Buf> bufs;
  std::vector<Op> ops;
  float* head_w = nullptr;
  float* head_b = nullptr;
  int gate_scratch = -1;            // AttentionUnet: buffer for the CUDA-core fallback of the gate GEMM
  int acc_scratch = -1;             // 3D nets: the first block's output buffer, dead after encode2, as fp32 scratch for K-split blocks
  int pool_scratch = -1;            // UNet3D: a level-0 decoder buffer, idle during the encoder, that takes the (y, x)-pooled
                                    // planes the row kernel's epilogue writes before the z pairs are reduced
  std::vector<void*> dev_allocs;

  // Siam_UNet, 'single' normalisation: frame t is the current frame of pair t and the previous frame of pair t + 1, and
  // its encoder output is the same in both. siam_shared = tiles per frame (> 0) runs the twin encoder ONCE over the
  // B + siam_shared unique tiles of a batch of B consecutive pairs [previous frame of the first pair | current frames]
  // instead of over 2 B: the previous stream is images [0, B), the current stream images [siam_shared, siam_shared + B).
  int siam_shared = 0;
  // plan
  int B = 0, D = 1, H = 0, W = 0;
  size_t ws_bytes = 0;

  int force_direct = 0;             // debugging: run every conv on the CUDA-core kernels
  int no_fuse = 0;                  // debugging: keep the max-pool as its own kernel
  int profile = 0;                  // bracket every op with CUDA events
  int debug_stop = -1;              // test hook: >= 0 ends net_forward after that op (-1: run the whole program)
  bool stopped = false;             // the last forward ended at debug_stop (its profile events are incomplete)
  std::vector<cudaEvent_t> events;  // 2 per op
  std::vector<int> op_kinds;        // kind (+16 if it ran on the CUDA-core fallback) of the last forward
};

int net_build(Net* n);                       // program + layer table from kind/nf/...
int net_finalize(Net* n);                    // fold, pack, upload
long long net_plan(Net* n, int B, int D, int H, int W);   // returns workspace bytes, <0 on error
int net_forward(Net* n, const void* in, int in_kind, const void* in2, float* out_val, uint8_t* out_u8,
                void* workspace, cudaStream_t stream);
int net_debug_copy(Net* n, const char* buf_name, void* workspace, void* dst_host, long long max_bytes);
int net_profile_read(Net* n, int max_ops, int* kinds, float* ms, int* n_ops);
void net_destroy(Net* n);

}  // namespace biu
