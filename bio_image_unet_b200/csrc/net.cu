// Layer programs of the reference's model families and their execution on a batch of tiles.
//   Unet          unet/unet.py:16-104            (2D, depth 4)
//   Siam_UNet     siam_unet/siam_unet.py:18-148  (twin encoder, shared weights)
//   UNet3D        unet3d/unet3d.py:18-99         (3D, depth 3)
//   MultiOutputUnet3D  multi_output_unet3d/multi_output_unet3d.py:13-170
//   MultiOutputNestedUNet(_3Levels)  multi_output_unet/multi_output_nested_unet.py:58-240  (U-Net++, dense skips)
// Activations are NHWC / NDHWC with channel counts padded to 16; torch.cat((up, skip), 1) is replaced by
// writing both producers into one buffer at channel offsets.
#include "net.h"
#include "common.cuh"
#include "conv_tc.cuh"

#include <cmath>
#include <cstring>

namespace biu {

static int pad16(int c) { return (c + 15) / 16 * 16; }

static float host_round_tf32(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  if ((u & 0x7F800000u) == 0x7F800000u) return v;
  u += 0x1000u;            // round to nearest, ties away (cvt.rna)
  u &= 0xFFFFE000u;
  memcpy(&v, &u, 4);
  return v;
}
static uint16_t host_bf16(float v) {
  uint32_t u;
  memcpy(&u, &v, 4);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7FFFu + ((u >> 16) & 1u);   // round to nearest even
  return (uint16_t)(u >> 16);
}
static uint16_t host_fp16(float v) {
  const __half_raw r = __float2half_rn(v);   // round to nearest even; beyond +-65504 -> +-inf
  return r.x;
}

struct Builder {
  Net* n;
  int buf(const std::string& name, int level, int ctot, int batch_mul = 1) {
    Buf b;
    b.level = level; b.ctot = ctot; b.batch_mul = batch_mul; b.name = name;
    n->bufs.push_back(b);
    return (int)n->bufs.size() - 1;
  }
  int conv_layer(const std::string& name, std::vector<Segment> segs, int cin_phys, int cout, int k) {
    ConvLayer L;
    L.name = name;
    L.segs = segs;
    L.cin_log = 0;
    for (auto& s : segs) L.cin_log += s.count;
    L.cin_phys = cin_phys;
    L.cout = cout;
    L.cout_pad = pad16(cout);
    L.kw = L.kh = k;
    L.kd = n->dims == 3 ? k : 1;
    n->layers.push_back(L);
    return (int)n->layers.size() - 1;
  }
  int up_layer(const std::string& name, int cin, int cout) {
    ConvLayer L;
    L.name = name;
    L.segs = {{0, cin, 0}};
    L.cin_log = cin; L.cin_phys = pad16(cin);
    L.cout = cout; L.cout_pad = pad16(cout);
    L.is_up = true;
    L.nq = n->dims == 3 ? 8 : 4;
    n->layers.push_back(L);
    return (int)n->layers.size() - 1;
  }
  // AttentionBlock(F_g = F_l = c, n_coefficients = nc) reading the concat buffer [up (gate) | skip]
  int gate_layer(const std::string& name, int c, int nc) {
    ConvLayer L;
    L.name = name;
    L.segs = {{0, c, 0}, {c, c, pad16(c)}};
    L.cin_log = 2 * c; L.cin_phys = 2 * pad16(c);
    L.cout = nc; L.cout_pad = pad16(nc);
    L.is_gate = true;
    L.slope = 0.f;
    n->layers.push_back(L);
    return (int)n->layers.size() - 1;
  }
  void op(OpKind kind, int layer, int src, int src_coff, int dst, int dst_coff, int c, int level, int batch_mul = 1,
          int src_img0 = 0, int dst_img0 = 0, int pool_mode = 0) {
    Op o;
    o.kind = kind; o.layer = layer; o.src = src; o.src_coff = src_coff; o.dst = dst; o.dst_coff = dst_coff;
    o.c = c; o.level = level; o.batch_mul = batch_mul; o.src_img0 = src_img0; o.dst_img0 = dst_img0;
    o.pool_mode = pool_mode;
    n->ops.push_back(o);
  }
  // plain block: src buffer (dense, logical channels = cin) -> dst
  void block(const std::string& name, int src, int cin, int dst, int dst_coff, int cout, int level, int bm = 1) {
    int L = conv_layer(name, {{0, cin, 0}}, pad16(cin), cout, 3);
    op(OP_CONV, L, src, 0, dst, dst_coff, pad16(cin), level, bm);
  }
  // block reading a concat buffer [up | skip]
  void block_cat(const std::string& name, int src, int c_up, int c_skip, int dst, int cout, int level) {
    int L = conv_layer(name, {{0, c_up, 0}, {c_up, c_skip, pad16(c_up)}}, pad16(c_up) + pad16(c_skip), cout, 3);
    op(OP_CONV, L, src, 0, dst, 0, pad16(c_up) + pad16(c_skip), level);
  }
};

int net_build(Net* n) {
  n->layers.clear(); n->bufs.clear(); n->ops.clear();
  Builder b{n};
  const int nf = n->nf;
  n->head_total = 0;
  for (int c : n->head_channels) n->head_total += c;
  BIU_REQUIRE(n->head_total >= 1 && n->head_total <= kMaxHead, "between 1 and %d output channels supported (got %d)",
              kMaxHead, n->head_total);
  BIU_REQUIRE(nf >= 2 && nf % 2 == 0, "n_filter must be even (got %d)", nf);

  if (n->kind == NET_UNET2D || n->kind == NET_SIAM2D || n->kind == NET_UNET2D_V0 || n->kind == NET_ATTUNET2D ||
      n->kind == NET_MO2D) {      // NET_MO2D: Unet body, heads 'output_layers.<name>' (multi_output_unet.py:62-65)
    n->dims = 2;
    n->levels = 4;
    const bool siam = n->kind == NET_SIAM2D;
    const bool v0 = n->kind == NET_UNET2D_V0;       // unet/unet_v0.py: ReLU blocks, skips after the first conv, decode9
    const bool att = n->kind == NET_ATTUNET2D;      // unet/attention_unet.py: gated skips, cat((attention, up))
    BIU_REQUIRE(!att || nf % 2 == 0, "AttentionUnet needs an even n_filter");
    // 'control' ignores the previous frame (siam_unet.py:122-123): its encoder pass is dead work and is skipped
    const int bm = (siam && n->siam_mode != SIAM_CONTROL) ? 2 : 1;
    int ch[5] = {nf, 2 * nf, 4 * nf, 8 * nf, 16 * nf};
    int e_a[4], cat[4], m[4], d_a[4], d_b[4];
    for (int l = 0; l < 4; ++l) {
      e_a[l] = b.buf("e" + std::to_string(2 * l + 1), l, pad16(ch[l]), bm);
      cat[l] = b.buf("cat" + std::to_string(4 - l), l, 2 * pad16(ch[l]), bm);
      m[l] = b.buf("m" + std::to_string(l + 1), l + 1, pad16(ch[l]), bm);
    }
    int join = -1, joincat = -1;
    if (siam && n->siam_mode == SIAM_CONCAT) joincat = b.buf("joincat", 4, 2 * pad16(ch[3]));
    if (siam && n->siam_mode != SIAM_CONTROL) join = b.buf("join", 4, pad16(ch[3]));
    int mid1 = b.buf("mid1", 4, pad16(ch[4]));
    int mid2 = b.buf("mid2", 4, pad16(ch[4]));
    int psi[4] = {-1, -1, -1, -1}, gate_scratch = -1;
    for (int l = 3; l >= 0; --l) {
      d_a[l] = b.buf("d" + std::to_string(2 * (3 - l) + 1), l, pad16(ch[l]));
      d_b[l] = (l > 0 || v0) ? b.buf("d" + std::to_string(2 * (3 - l) + 2), l, pad16(ch[l])) : -1;
      if (att) psi[l] = b.buf("psi" + std::to_string(4 - l), l, 4 / fmt_esz(n->fmt));      // one float per pixel
    }
    if (att) gate_scratch = b.buf("gate_scratch", 0, pad16(nf / 2));              // CUDA-core fallback only
    n->gate_scratch = gate_scratch;
    // encoder
    for (int l = 0; l < 4; ++l) {
      const std::string n1 = "encode" + std::to_string(2 * l + 1), n2 = "encode" + std::to_string(2 * l + 2);
      // the skip tensor lives in the upper half of the level's concat buffer: the second conv's output
      // (unet/unet.py:72-83), or the FIRST conv's for Unet_v0 (unet/unet_v0.py:91-103)
      const int c1_dst = v0 ? cat[l] : e_a[l], c1_coff = v0 ? pad16(ch[l]) : 0;
      if (l == 0) {
        int L = b.conv_layer(n1, {{0, n->in_ch, 0}}, n->in_ch, ch[0], 3);
        b.op(OP_FIRST, L, -1, 0, c1_dst, c1_coff, n->in_ch, 0, 1, 0, 0);
        if (bm == 2) b.op(OP_FIRST, L, -2, 0, c1_dst, c1_coff, n->in_ch, 0, 1, 0, 1);
      } else {
        int L = b.conv_layer(n1, {{0, ch[l - 1], 0}}, pad16(ch[l - 1]), ch[l], 3);
        b.op(OP_CONV, L, m[l - 1], 0, c1_dst, c1_coff, pad16(ch[l - 1]), l, bm);
      }
      {
        int L = b.conv_layer(n2, {{0, ch[l], 0}}, pad16(ch[l]), ch[l], 3);
        if (v0) b.op(OP_CONV, L, cat[l], pad16(ch[l]), e_a[l], 0, pad16(ch[l]), l, bm);
        else b.op(OP_CONV, L, e_a[l], 0, cat[l], pad16(ch[l]), pad16(ch[l]), l, bm);
      }
      if (v0) {
        b.op(OP_POOL, -1, e_a[l], 0, m[l], 0, pad16(ch[l]), l, bm);
      } else if (l < 3 || !siam || n->siam_mode != SIAM_CONCAT) {
        b.op(OP_POOL, -1, cat[l], pad16(ch[l]), m[l], 0, pad16(ch[l]), l, bm);
      } else {  // concat join: pooled current -> channels [0, 8nf), pooled previous -> [8nf, 16nf)
        b.op(OP_POOL, -1, cat[l], pad16(ch[l]), joincat, 0, pad16(ch[l]), l, 1, 0, 0);
        b.op(OP_POOL, -1, cat[l], pad16(ch[l]), joincat, pad16(ch[l]), pad16(ch[l]), l, 1, 1, 0);
      }
    }
    int mid_src = m[3];
    if (siam && n->siam_mode == SIAM_CONCAT) {
      int L = b.conv_layer("conv_concat", {{0, ch[3], 0}, {ch[3], ch[3], pad16(ch[3])}}, 2 * pad16(ch[3]), ch[3], 3);
      b.op(OP_CONV, L, joincat, 0, join, 0, 2 * pad16(ch[3]), 4);
      mid_src = join;
    } else if (siam && (n->siam_mode == SIAM_MAX || n->siam_mode == SIAM_CORR)) {
      // max: element-wise maximum; corr: depth-wise cross-correlation of the two embeddings (siam_unet.py:75-83,114-117)
      Op o; o.kind = n->siam_mode == SIAM_MAX ? OP_MAXJOIN : OP_XCORR;
      o.src = m[3]; o.dst = join; o.c = pad16(ch[3]); o.level = 4; o.src2 = 1;
      n->ops.push_back(o);
      mid_src = join;
    }
    b.block("middle_conv1", mid_src, ch[3], mid1, 0, ch[4], 4);
    b.block("middle_conv2", mid1, ch[4], mid2, 0, ch[4], 4);
    // decoder
    int prev = mid2, prev_c = ch[4];
    for (int l = 3; l >= 0; --l) {
      const int k = 3 - l;  // 0..3
      int U = b.up_layer("up" + std::to_string(k + 1), prev_c, ch[l]);
      b.op(OP_UP, U, prev, 0, cat[l], 0, pad16(prev_c), l + 1);
      if (att) {
        // a = skip * psi(up, skip) in place, then decode(cat((a, up))) (unet/attention_unet.py:88-90): the
        // block's logical channels [0, C) are the gated skip (physical upper half), [C, 2C) the up-sampled tensor
        int G = b.gate_layer("attention" + std::to_string(k + 1), ch[l], ch[l] / 2);
        b.op(OP_GATE, G, cat[l], 0, psi[l], 0, 2 * pad16(ch[l]), l);
        b.op(OP_MULPSI, -1, psi[l], 0, cat[l], pad16(ch[l]), pad16(ch[l]), l);
        int L = b.conv_layer("decode" + std::to_string(2 * k + 1), {{0, ch[l], pad16(ch[l])}, {ch[l], ch[l], 0}},
                             2 * pad16(ch[l]), ch[l], 3);
        b.op(OP_CONV, L, cat[l], 0, d_a[l], 0, 2 * pad16(ch[l]), l);
      } else {
        b.block_cat("decode" + std::to_string(2 * k + 1), cat[l], ch[l], ch[l], d_a[l], ch[l], l);
      }
      if (l > 0 || v0) {
        b.block("decode" + std::to_string(2 * k + 2), d_a[l], ch[l], d_b[l], 0, ch[l], l);
        prev = d_b[l]; prev_c = ch[l];
      } else {
        int L = b.conv_layer("decode8", {{0, ch[0], 0}}, pad16(ch[0]), ch[0], 3);
        b.op(OP_CONV_HEAD, L, d_a[0], 0, -1, 0, pad16(ch[0]), 0);
      }
    }
    if (v0) {     // decode9: 3x3 block n_filter -> 1, then the 1x1 head 1 -> 1 (unet/unet_v0.py:49-52,104-105)
      int L = b.conv_layer("decode9", {{0, ch[0], 0}}, pad16(ch[0]), 1, 3);
      b.op(OP_CONV_HEAD, L, d_b[0], 0, -1, 0, pad16(ch[0]), 0);
      for (auto& L2 : n->layers) L2.slope = 0.f;                       // every block of Unet_v0 is Conv-BN-ReLU
    }
  } else if (n->kind == NET_UNET3D || n->kind == NET_MO3D) {
    n->dims = 3;
    n->levels = 3;
    const bool interp = n->use_interp != 0;
    const bool tri = n->kind == NET_UNET3D && interp;       // UNet3D(use_interpolation=True): trilinear x2, no up-conv
    const int h = nf / 2;
    // level l: first conv a[l] -> b[l] channels, second -> c[l]
    int c_in[4] = {n->in_ch, nf, 2 * nf, 4 * nf};
    int c_a[4] = {h, nf, 2 * nf, 4 * nf};
    int c_b[4] = {nf, 2 * nf, 4 * nf, 8 * nf};
    int up_c[3] = {2 * nf, 4 * nf, 8 * nf};          // channels of the upsampled tensor arriving at level l
    int e_a[3], cat[3], m[3];
    for (int l = 0; l < 3; ++l) {
      e_a[l] = b.buf("e" + std::to_string(2 * l + 1), l, pad16(c_a[l]));
      cat[l] = b.buf("cat" + std::to_string(3 - l), l, pad16(up_c[l]) + pad16(c_b[l]));
      m[l] = b.buf("m" + std::to_string(l + 1), l + 1, pad16(c_b[l]));
    }
    int mid1 = b.buf("mid1", 3, pad16(c_a[3]));
    int mid2 = b.buf("mid2", 3, pad16(c_b[3]));
    int dec_out[3] = {h, 2 * nf, 4 * nf};             // decode6 / decode4 / decode2 outputs
    int dec_mid[3] = {nf, 2 * nf, 4 * nf};            // decode5 / decode3 / decode1 outputs
    int d_a[3], d_b[3], upt[3];
    for (int l = 2; l >= 0; --l) {
      d_a[l] = b.buf("d" + std::to_string(2 * (2 - l) + 1), l, pad16(dec_mid[l]));
      d_b[l] = l > 0 ? b.buf("d" + std::to_string(2 * (2 - l) + 2), l, pad16(dec_out[l])) : -1;
      upt[l] = (interp && !tri) ? b.buf("upn" + std::to_string(3 - l), l, pad16(up_c[l])) : -1;
    }
    if (pad16(dec_mid[0]) >= pad16(c_b[0])) n->pool_scratch = d_a[0];
    n->acc_scratch = e_a[0];
    for (int l = 0; l < 3; ++l) {
      const std::string n1 = "encode" + std::to_string(2 * l + 1), n2 = "encode" + std::to_string(2 * l + 2);
      if (l == 0) {
        int L = b.conv_layer(n1, {{0, n->in_ch, 0}}, n->in_ch, c_a[0], 3);
        b.op(OP_FIRST, L, -1, 0, e_a[0], 0, n->in_ch, 0);
      } else {
        b.block(n1, m[l - 1], c_in[l], e_a[l], 0, c_a[l], l);
      }
      b.block(n2, e_a[l], c_a[l], cat[l], pad16(up_c[l]), c_b[l], l);
      b.op(OP_POOL, -1, cat[l], pad16(up_c[l]), m[l], 0, pad16(c_b[l]), l, 1, 0, 0, (interp && !tri) ? 1 : 0);
    }
    b.block("middle_conv1", m[2], c_in[3], mid1, 0, c_a[3], 3);
    b.block("middle_conv2", mid1, c_a[3], mid2, 0, c_b[3], 3);
    int prev = mid2, prev_c = c_b[3];
    for (int l = 2; l >= 0; --l) {
      const int k = 2 - l;
      if (tri) {               // F.interpolate(scale_factor=2, mode='trilinear', align_corners=False), unet3d.py:78-92
        b.op(OP_UPTRILINEAR, -1, prev, 0, cat[l], 0, pad16(prev_c), l + 1);
      } else if (!interp) {
        int U = b.up_layer("up" + std::to_string(k + 1), prev_c, prev_c);
        b.op(OP_UP, U, prev, 0, cat[l], 0, pad16(prev_c), l + 1);
      } else {
        b.op(OP_UPNEAREST, -1, prev, 0, upt[l], 0, pad16(prev_c), l + 1);
        b.block("up" + std::to_string(k + 1) + "_conv", upt[l], prev_c, cat[l], 0, prev_c, l);
      }
      b.block_cat("decode" + std::to_string(2 * k + 1), cat[l], up_c[l], c_b[l], d_a[l], dec_mid[l], l);
      if (l > 0) {
        b.block("decode" + std::to_string(2 * k + 2), d_a[l], dec_mid[l], d_b[l], 0, dec_out[l], l);
        prev = d_b[l]; prev_c = dec_out[l];
      } else {
        int L = b.conv_layer("decode6", {{0, dec_mid[0], 0}}, pad16(dec_mid[0]), dec_out[0], 3);
        b.op(OP_CONV_HEAD, L, d_a[0], 0, -1, 0, pad16(dec_mid[0]), 0);
      }
    }
  } else if (n->kind == NET_NESTED2D || n->kind == NET_NESTED2D_3L) {
    // U-Net++ (multi_output_unet/multi_output_nested_unet.py:58-148 / :151-240): node x{l}_{j} = VGGBlock(cat(x{l}_0 ..
    // x{l}_{j-1}, up(x{l+1}_{j-1}))), VGGBlock = (Conv3x3 - BatchNorm - LeakyReLU(0.1)) x 2, up = bilinear x2 with
    // align_corners=True. All nodes of a level live in ONE buffer: physical channels [0, 2 C_l) hold the up-sampled
    // tensor of the block being computed (always 128-byte aligned for the up-sampling kernel's stores), node j
    // follows at 2 C_l + j C_l, so every torch.cat is a channel PREFIX of the buffer (the layer's segment table maps
    // the reference's logical channel order onto it) and nothing is ever copied.
    n->dims = 2;
    const int Lv = n->kind == NET_NESTED2D ? 4 : 3;
    n->levels = Lv;
    int ch[5], pc[5], upw[5], dense[5], mid[5], m[5];
    for (int l = 0; l <= Lv; ++l) { ch[l] = nf << l; pc[l] = pad16(ch[l]); }
    for (int l = 0; l <= Lv; ++l) upw[l] = l < Lv ? pc[l + 1] : 0;      // width of the level's up-sampling slot
    for (int l = 0; l <= Lv; ++l) {
      const int J = Lv - l;                              // nodes x{l}_0 .. x{l}_J; x0_J feeds the heads only
      dense[l] = b.buf("x" + std::to_string(l), l, upw[l] + (l == 0 ? J : J + 1) * pc[l]);
      mid[l] = b.buf("v" + std::to_string(l), l, pc[l]);
      m[l] = l < Lv ? b.buf("m" + std::to_string(l + 1), l + 1, pc[l]) : -1;
    }
    auto vgg_conv = [&](const std::string& node, int which, std::vector<Segment> segs, int cin_phys, int cout) {
      int L = b.conv_layer(node, segs, cin_phys, cout, 3);
      n->layers[L].conv_key = node + ".conv" + std::to_string(which);
      n->layers[L].bn_key = node + ".bn" + std::to_string(which);
      return L;
    };
    for (int s = 0; s <= Lv; ++s) {
      {   // backbone node x{s}_0
        const std::string node = "conv" + std::to_string(s) + "_0";
        if (s == 0) {
          int L = vgg_conv(node, 1, {{0, n->in_ch, 0}}, n->in_ch, ch[0]);
          b.op(OP_FIRST, L, -1, 0, mid[0], 0, n->in_ch, 0);
        } else {
          int L = vgg_conv(node, 1, {{0, ch[s - 1], 0}}, pc[s - 1], ch[s]);
          b.op(OP_CONV, L, m[s - 1], 0, mid[s], 0, pc[s - 1], s);
        }
        int L2 = vgg_conv(node, 2, {{0, ch[s], 0}}, pc[s], ch[s]);
        b.op(OP_CONV, L2, mid[s], 0, dense[s], upw[s], pc[s], s);
        if (s < Lv) b.op(OP_POOL, -1, dense[s], upw[s], m[s], 0, pc[s], s);
      }
      for (int j = 1; j <= s; ++j) {
        const int l = s - j;
        const std::string node = "conv" + std::to_string(l) + "_" + std::to_string(j);
        b.op(OP_UPBILINEAR, -1, dense[l + 1], upw[l + 1] + (j - 1) * pc[l + 1], dense[l], 0, pc[l + 1], l + 1);
        std::vector<Segment> segs;
        for (int k = 0; k < j; ++k) segs.push_back({k * ch[l], ch[l], upw[l] + k * pc[l]});
        segs.push_back({j * ch[l], ch[l + 1], 0});
        const int cin_phys = upw[l] + j * pc[l];
        int L = vgg_conv(node, 1, segs, cin_phys, ch[l]);
        b.op(OP_CONV, L, dense[l], 0, mid[l], 0, cin_phys, l);
        int L2 = vgg_conv(node, 2, {{0, ch[l], 0}}, pc[l], ch[l]);
        if (l == 0 && j == Lv) b.op(OP_CONV_HEAD, L2, mid[0], 0, -1, 0, pc[0], 0);
        else b.op(OP_CONV, L2, mid[l], 0, dense[l], upw[l] + j * pc[l], pc[l], l);
      }
    }
  } else {
    BIU_REQUIRE(false, "unknown network kind %d", n->kind);
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
static const HostTensor* find_param(Net* n, const std::string& name) {
  auto it = n->params.find(name);
  return it == n->params.end() ? nullptr : &it->second;
}

template <typename T>
static int upload(Net* n, const std::vector<T>& h, T** dptr) {
  void* d = nullptr;
  BIU_CHECK_CUDA(cudaMalloc(&d, h.size() * sizeof(T) + 16));
  BIU_CHECK_CUDA(cudaMemcpy(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
  n->dev_allocs.push_back(d);
  *dptr = reinterpret_cast<T*>(d);
  return 0;
}

// Tensor-core weights: `h` is laid out in the target order; it is converted to the net's format (bf16 / fp16, or fp32
// rounded to tf32) and uploaded.
static int upload_packed(Net* n, const std::vector<float>& h, void** dptr) {
  if (n->fmt == FMT_TF32) {
    std::vector<float> wp(h.size());
    for (size_t i = 0; i < h.size(); ++i) wp[i] = host_round_tf32(h[i]);
    float* d = nullptr;
    if (upload(n, wp, &d)) return -1;
    *dptr = d;
    return 0;
  }
  BIU_REQUIRE(n->fmt == FMT_BF16 || n->fmt == FMT_F16, "no tensor-core weights in element format %d", n->fmt);
  std::vector<uint16_t> wp(h.size());
  for (size_t i = 0; i < h.size(); ++i) wp[i] = n->fmt == FMT_F16 ? host_fp16(h[i]) : host_bf16(h[i]);
  uint16_t* d = nullptr;
  if (upload(n, wp, &d)) return -1;
  *dptr = d;
  return 0;
}

// A convolution with bias followed by BatchNorm (eval), by state_dict prefixes.
struct ConvBn {
  const HostTensor *w, *bias, *g, *be, *mu, *var;
};
static bool find_conv_bn(Net* n, const std::string& conv, const std::string& bn, ConvBn* p) {
  p->w = find_param(n, conv + ".weight");
  p->bias = find_param(n, conv + ".bias");
  p->g = find_param(n, bn + ".weight");
  p->be = find_param(n, bn + ".bias");
  p->mu = find_param(n, bn + ".running_mean");
  p->var = find_param(n, bn + ".running_var");
  return p->w && p->bias && p->g && p->be && p->mu && p->var;
}
// Output channel c of BN(conv(x) + b) = sc * conv(x) + shift, in float64: sc = g / sqrt(var + 1e-5),
// shift = be + (b - mu) * sc.
static void fold_bn(const ConvBn& p, int c, double* sc, double* shift) {
  *sc = (double)p.g->data[c] / std::sqrt((double)p.var->data[c] + 1e-5);
  *shift = (double)p.be->data[c] + ((double)p.bias->data[c] - (double)p.mu->data[c]) * *sc;
}

int net_finalize(Net* n) {
  const bool tc = n->fmt != FMT_F32;          // the tensor-core modes pack weights for the tcgen05 kernels
  for (auto& L : n->layers) {
    const int taps = L.kd * L.kh * L.kw;
    if (L.is_gate) {
      // AttentionBlock (unet/attention_unet.py:143-181): g1 + x1 = BN(conv1x1(gate)) + BN(conv1x1(skip)) is one GEMM
      // over the concat buffer with the BatchNorm scales folded into the weights (fp64 on the host), ReLU, then
      // psi = sigmoid(BN(conv1x1)) as a 1x1 head with BatchNorm(1) folded into its weight and bias.
      const int c = L.cin_log / 2;
      const char* br[2] = {".W_gate", ".W_x"};
      std::vector<float> wd((size_t)L.cin_phys * L.cout_pad, 0.f);
      std::vector<float> scale(L.cout_pad, 1.f), shift(L.cout_pad, 0.f);
      for (int s2 = 0; s2 < 2; ++s2) {
        const std::string base = L.name + br[s2];
        ConvBn p;
        BIU_REQUIRE(find_conv_bn(n, base + ".0", base + ".1", &p), "state_dict is missing parameters of '%s'", base.c_str());
        BIU_REQUIRE((long long)p.w->data.size() == (long long)L.cout * c, "'%s.0.weight' has %lld elements, expected %lld",
                    base.c_str(), (long long)p.w->data.size(), (long long)L.cout * c);
        for (int co = 0; co < L.cout; ++co) {
          double sc, sh;
          fold_bn(p, co, &sc, &sh);
          shift[co] += (float)sh;
          for (int ci = 0; ci < c; ++ci)
            wd[(size_t)(L.segs[s2].pstart + ci) * L.cout_pad + co] = (float)(sc * (double)p.w->data[(size_t)co * c + ci]);
        }
      }
      if (upload(n, wd, &L.w_direct)) return -1;
      if (upload(n, scale, &L.scale)) return -1;
      if (upload(n, shift, &L.shift)) return -1;
      if (tc) {
        std::vector<float> wp((size_t)L.cout_pad * L.cin_phys, 0.f);
        for (int co = 0; co < L.cout; ++co)
          for (int ci = 0; ci < L.cin_phys; ++ci) wp[(size_t)co * L.cin_phys + ci] = wd[(size_t)ci * L.cout_pad + co];
        if (int rc = upload_packed(n, wp, &L.w_tc)) return rc;
      }
      {
        const std::string base = L.name + ".psi";
        ConvBn p;
        BIU_REQUIRE(find_conv_bn(n, base + ".0", base + ".1", &p), "state_dict is missing parameters of '%s'", base.c_str());
        BIU_REQUIRE((long long)p.w->data.size() == (long long)L.cout, "'%s.0.weight' has %lld elements, expected %d",
                    base.c_str(), (long long)p.w->data.size(), L.cout);
        double sc, sh;
        fold_bn(p, 0, &sc, &sh);
        std::vector<float> gw(L.cout_pad, 0.f), gb(1, (float)sh);
        for (int co = 0; co < L.cout; ++co) gw[co] = (float)(sc * (double)p.w->data[co]);
        if (upload(n, gw, &L.gate_w)) return -1;
        if (upload(n, gb, &L.gate_b)) return -1;
      }
      continue;
    }
    if (!L.is_up) {
      const std::string ck = L.conv_key.empty() ? L.name + ".0" : L.conv_key;
      const std::string bk = L.bn_key.empty() ? L.name + ".1" : L.bn_key;
      ConvBn p;
      BIU_REQUIRE(find_conv_bn(n, ck, bk, &p), "state_dict is missing parameters of block '%s' / '%s'", ck.c_str(),
                  bk.c_str());
      const HostTensor* w = p.w;
      BIU_REQUIRE((long long)w->data.size() == (long long)L.cout * L.cin_log * taps,
                  "'%s.weight' has %lld elements, expected %lld", ck.c_str(), (long long)w->data.size(),
                  (long long)L.cout * L.cin_log * taps);
      std::vector<float> scale(L.cout_pad, 0.f), shift(L.cout_pad, 0.f);
      for (int co = 0; co < L.cout; ++co) {
        double sc, sh;
        fold_bn(p, co, &sc, &sh);
        scale[co] = (float)sc;
        shift[co] = (float)sh;
      }
      // physical channel of every logical input channel
      std::vector<int> phys(L.cin_log);
      for (auto& sg : L.segs)
        for (int i = 0; i < sg.count; ++i) phys[sg.lstart + i] = sg.pstart + i;
      std::vector<float> wd((size_t)taps * L.cin_phys * L.cout_pad, 0.f);
      for (int co = 0; co < L.cout; ++co)
        for (int ci = 0; ci < L.cin_log; ++ci)
          for (int t = 0; t < taps; ++t)
            wd[((size_t)t * L.cin_phys + phys[ci]) * L.cout_pad + co] = w->data[((size_t)co * L.cin_log + ci) * taps + t];
      if (upload(n, wd, &L.w_direct)) return -1;
      if (upload(n, scale, &L.scale)) return -1;
      if (upload(n, shift, &L.shift)) return -1;
      // first block of a 2D net (one input channel): packing for the row kernel's first mode - the dx taps are the K
      // dimension (zero padded to 16 bf16 / fp16 or 8 tf32 elements), the dy taps are folded into N in the order dy = 2, 1, 0
      if (tc && L.cin_log == 1 && L.kd == 1 && L.kw == 3 && L.kh == 3 && (L.cout_pad == 16 || L.cout_pad == 32)) {
        const int kel = 32 / fmt_esz(n->fmt), nfold = 3 * L.cout_pad;
        std::vector<float> wf((size_t)nfold * kel, 0.f);
        for (int dy = 0; dy < 3; ++dy)
          for (int dx = 0; dx < 3; ++dx)
            for (int co = 0; co < L.cout; ++co)
              wf[((size_t)(2 - dy) * L.cout_pad + co) * kel + dx] = w->data[(size_t)co * taps + dy * 3 + dx];
        if (int rc = upload_packed(n, wf, &L.w_first)) return rc;
        std::vector<float> s255(L.cout_pad, 0.f);
        for (int co = 0; co < L.cout; ++co) s255[co] = scale[co] / 255.0f;
        if (upload(n, s255, &L.scale_first)) return -1;
      }
      if (tc && L.cin_phys % 16 == 0) {
        std::vector<float> wp((size_t)taps * L.cout_pad * L.cin_phys, 0.f);
        for (int t = 0; t < taps; ++t)
          for (int co = 0; co < L.cout; ++co)
            for (int ci = 0; ci < L.cin_log; ++ci)
              wp[((size_t)t * L.cout_pad + co) * L.cin_phys + phys[ci]] = w->data[((size_t)co * L.cin_log + ci) * taps + t];
        if (int rc = upload_packed(n, wp, &L.w_tc)) return rc;
        // narrow blocks (Cout <= 32): second packing with the dy taps folded into the GEMM's N, in the order
        // dy = 2, 1, 0 = output rows r-1, r, r+1 of input row r (conv_rows.cuh)
        if (L.kw == 3 && (L.cout_pad <= 32 || (L.cout_pad == 64 && L.kd == 1 && fmt_esz(n->fmt) == 2))) {
          const int tz = L.kd * 3, nfold = 3 * L.cout_pad;
          std::vector<float> wf((size_t)tz * nfold * L.cin_phys, 0.f);
          for (int dz = 0; dz < L.kd; ++dz)
            for (int dy = 0; dy < 3; ++dy)
              for (int dx = 0; dx < 3; ++dx) {
                const int t = (dz * 3 + dy) * 3 + dx;
                for (int co = 0; co < L.cout; ++co)
                  for (int ci = 0; ci < L.cin_log; ++ci)
                    wf[((size_t)(dz * 3 + dx) * nfold + (2 - dy) * L.cout_pad + co) * L.cin_phys + phys[ci]] =
                        w->data[((size_t)co * L.cin_log + ci) * taps + t];
              }
          if (int rc = upload_packed(n, wf, &L.w_fold)) return rc;
          // 3D: third packing with the dz taps folded instead (planes narrower than 128 px: the row kernel's plane
          // mode streams the planes of a 16 x 8 tile), order dz = 2, 1, 0 = output planes z-1, z, z+1 of input plane z
          if (L.kd == 3 && L.cout_pad <= 32) {
            std::vector<float> wz((size_t)9 * nfold * L.cin_phys, 0.f);
            for (int dz = 0; dz < 3; ++dz)
              for (int dy = 0; dy < 3; ++dy)
                for (int dx = 0; dx < 3; ++dx) {
                  const int t = (dz * 3 + dy) * 3 + dx;
                  for (int co = 0; co < L.cout; ++co)
                    for (int ci = 0; ci < L.cin_log; ++ci)
                      wz[((size_t)(dy * 3 + dx) * nfold + (2 - dz) * L.cout_pad + co) * L.cin_phys + phys[ci]] =
                          w->data[((size_t)co * L.cin_log + ci) * taps + t];
                }
            if (int rc = upload_packed(n, wz, &L.w_fold_z)) return rc;
          }
        }
      }
    } else {
      const HostTensor* w = find_param(n, L.name + ".weight");
      const HostTensor* bias = find_param(n, L.name + ".bias");
      BIU_REQUIRE(w && bias, "state_dict is missing parameters of '%s'", L.name.c_str());
      BIU_REQUIRE((long long)w->data.size() == (long long)L.cin_log * L.cout * L.nq,
                  "'%s.weight' has %lld elements, expected %lld", L.name.c_str(), (long long)w->data.size(),
                  (long long)L.cin_log * L.cout * L.nq);
      // torch layout [Cin][Cout][(2)][2][2]; q = (az*2 + ay)*2 + ax is the flattened kernel index
      std::vector<float> wd((size_t)L.nq * L.cin_phys * L.cout_pad, 0.f);
      std::vector<float> shift((size_t)L.nq * L.cout_pad, 0.f), scale((size_t)L.nq * L.cout_pad, 1.f);
      for (int q = 0; q < L.nq; ++q)
        for (int co = 0; co < L.cout; ++co) {
          shift[(size_t)q * L.cout_pad + co] = bias->data[co];
          for (int ci = 0; ci < L.cin_log; ++ci)
            wd[((size_t)q * L.cin_phys + ci) * L.cout_pad + co] = w->data[((size_t)ci * L.cout + co) * L.nq + q];
        }
      if (upload(n, wd, &L.w_direct)) return -1;
      if (upload(n, scale, &L.scale)) return -1;
      if (upload(n, shift, &L.shift)) return -1;
      if (tc) {
        std::vector<float> wp((size_t)L.nq * L.cout_pad * L.cin_phys, 0.f);
        for (int q = 0; q < L.nq; ++q)
          for (int co = 0; co < L.cout; ++co)
            for (int ci = 0; ci < L.cin_log; ++ci)
              wp[((size_t)q * L.cout_pad + co) * L.cin_phys + ci] = w->data[((size_t)ci * L.cout + co) * L.nq + q];
        if (int rc = upload_packed(n, wp, &L.w_tc)) return rc;
      }
    }
  }
  // head(s): 2D 'final.0', 3D 'final', multi-output 'output_layers.<name>'
  {
    const ConvLayer& last = n->layers[n->ops.back().layer];
    std::vector<float> hw((size_t)n->head_total * last.cout_pad, 0.f), hb(n->head_total, 0.f);
    int row = 0;
    for (size_t hi = 0; hi < n->head_channels.size(); ++hi) {
      std::string base;
      if (n->kind == NET_MO3D || n->kind == NET_MO2D || n->kind == NET_NESTED2D || n->kind == NET_NESTED2D_3L)
        base = "output_layers." + n->head_names[hi];
      else if (n->kind == NET_UNET3D) base = "final";
      else base = "final.0";
      const HostTensor* w = find_param(n, base + ".weight");
      const HostTensor* bias = find_param(n, base + ".bias");
      BIU_REQUIRE(w && bias, "state_dict is missing the head '%s'", base.c_str());
      BIU_REQUIRE((long long)w->data.size() == (long long)n->head_channels[hi] * last.cout,
                  "'%s.weight' has %lld elements, expected %lld", base.c_str(), (long long)w->data.size(),
                  (long long)n->head_channels[hi] * last.cout);
      for (int c = 0; c < n->head_channels[hi]; ++c, ++row) {
        for (int ci = 0; ci < last.cout; ++ci) hw[(size_t)row * last.cout_pad + ci] = w->data[(size_t)c * last.cout + ci];
        hb[row] = bias->data[c];
      }
    }
    if (upload(n, hw, &n->head_w)) return -1;
    if (upload(n, hb, &n->head_b)) return -1;
  }
  n->params.clear();
  n->finalized = true;
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
static void level_dims(const Net* n, int level, int* D, int* H, int* W) {
  *H = n->H >> level;
  *W = n->W >> level;
  *D = n->dims == 3 ? (n->D >> level) : 1;
}

long long net_plan(Net* n, int B, int D, int H, int W) {
  const int div = 1 << n->levels;
  BIU_REQUIRE(B >= 1, "batch must be positive");
  // unet/unet.py:62-67 raises 'concatenation failed: wrong dimensions' otherwise
  BIU_REQUIRE(H % div == 0 && W % div == 0 && (n->dims == 2 || D % div == 0),
              "concatenation failed: wrong dimensions (tile %dx%dx%d is not divisible by %d)", D, H, W, div);
  n->B = B; n->D = n->dims == 3 ? D : 1; n->H = H; n->W = W;
  size_t off = 0;
  for (auto& b : n->bufs) {
    int d, h, w;
    level_dims(n, b.level, &d, &h, &w);
    b.offset = off;
    const size_t imgs = (b.batch_mul == 2 && n->siam_shared > 0) ? (size_t)B + n->siam_shared : (size_t)B * b.batch_mul;
    size_t bytes = imgs * d * h * w * b.ctot * fmt_esz(n->fmt);
    off += (bytes + 1023) & ~(size_t)1023;
  }
  n->ws_bytes = off;
  return (long long)off;
}

template <int FMT>
__global__ void max_join_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out,
                                long long nvec) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nvec; i += (long long)gridDim.x * blockDim.x) {
    uint4 x = a[i], y = b[i], r;
    if (fmt_esz(FMT) == 2) {
      r = make_uint4(max_half2<FMT>(x.x, y.x), max_half2<FMT>(x.y, y.y), max_half2<FMT>(x.z, y.z), max_half2<FMT>(x.w, y.w));
    } else {
      const float* xp = reinterpret_cast<const float*>(&x);
      const float* yp = reinterpret_cast<const float*>(&y);
      float* rp = reinterpret_cast<float*>(&r);
#pragma unroll
      for (int k = 0; k < 4; ++k) rp[k] = fmaxf(xp[k], yp[k]);
    }
    out[i] = r;
  }
}

// Depth-wise cross-correlation of the current and previous embeddings (siam_unet/siam_unet.py:75-83):
// F.conv2d(curr.view(1, B*C, h, w), prev.view(B*C, 1, h, w), groups=B*C, padding='same'), i.e.
//   out[b, y, x, c] = sum_{i, j} curr[b, y + i - (h-1)/2, x + j - (w-1)/2, c] * prev[b, i, j, c]      (zero outside;
// for even extents PyTorch puts the extra padding at the far end). One block per (image, group of G channels):
// both planes staged in shared memory as fp32, fp32 accumulation, 4 x 4 pixel micro-tiles per thread.
template <typename T>
__global__ void __launch_bounds__(256) xcorr_join_kernel(const T* __restrict__ cur, const T* __restrict__ prev,
                                                         T* __restrict__ out, int h, int w, int ctot, int G,
                                                         int round_tf32) {
  extern __shared__ float sm[];
  float* s_cur = sm;                    // [h*w][G]
  float* s_prev = sm + (size_t)h * w * G;
  const int groups = ctot / G;
  const int b = blockIdx.x / groups, c0 = (blockIdx.x % groups) * G;
  const long long img = (long long)b * h * w * ctot;
  for (int i = threadIdx.x; i < h * w * G; i += blockDim.x) {
    const int pix = i / G, c = i - pix * G;
    s_cur[i] = (float)cur[img + (long long)pix * ctot + c0 + c];
    s_prev[i] = (float)prev[img + (long long)pix * ctot + c0 + c];
  }
  __syncthreads();
  const int pt = (h - 1) / 2, pl = (w - 1) / 2;
  for (int o = threadIdx.x; o < h * w * G; o += blockDim.x) {
    const int pix = o / G, c = o - pix * G;
    const int y = pix / w, x = pix - y * w;
    float acc = 0.f;
    const int i_lo = max(0, pt - y), i_hi = min(h, h + pt - y);      // 0 <= y + i - pt < h
    const int j_lo = max(0, pl - x), j_hi = min(w, w + pl - x);
    for (int i = i_lo; i < i_hi; ++i) {
      const float* cr = s_cur + ((size_t)(y + i - pt) * w + (x - pl)) * G + c;
      const float* pr = s_prev + (size_t)i * w * G + c;
      for (int j = j_lo; j < j_hi; ++j) acc = fmaf(cr[(size_t)j * G], pr[(size_t)j * G], acc);
    }
    if (sizeof(T) == 4 && round_tf32) { uint32_t u; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(acc)); acc = __uint_as_float(u); }
    out[img + (long long)pix * ctot + c0 + c] = (T)acc;
  }
}

// Trilinear x2 up-sampling, align_corners=False (unet3d/unet3d.py:78-92): source coordinate (o + 0.5) / 2 - 0.5
// clamped at 0, neighbours clamped at the far end; NDHWC, 16-byte channel vectors.
template <typename T, int VEC>
__global__ void __launch_bounds__(256) up_trilinear_kernel(const T* __restrict__ in, int in_ctot, int in_coff, int c,
                                                           int B, int D, int H, int W, T* __restrict__ out, int out_ctot,
                                                           int out_coff, int round_tf32) {
  const int oD = 2 * D, oH = 2 * H, oW = 2 * W, cv = c / VEC;
  const long long total = (long long)B * oD * oH * oW * cv;
  for (long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long long)gridDim.x * blockDim.x) {
    long long r = idx;
    const int ch = (int)(r % cv) * VEC; r /= cv;
    const int x = (int)(r % oW); r /= oW;
    const int y = (int)(r % oH); r /= oH;
    const int z = (int)(r % oD); r /= oD;
    const int b = (int)r;
    int i0[3], i1[3]; float l1[3];
    const int o3[3] = {z, y, x}, n3[3] = {D, H, W};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      float src = fmaxf(0.5f * ((float)o3[a] + 0.5f) - 0.5f, 0.f);
      i0[a] = (int)src; i1[a] = min(i0[a] + 1, n3[a] - 1); l1[a] = src - (float)i0[a];
    }
    float acc[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) acc[k] = 0.f;
#pragma unroll
    for (int dz = 0; dz < 2; ++dz)
#pragma unroll
      for (int dy = 0; dy < 2; ++dy)
#pragma unroll
        for (int dx = 0; dx < 2; ++dx) {
          const float wgt = (dz ? l1[0] : 1.f - l1[0]) * (dy ? l1[1] : 1.f - l1[1]) * (dx ? l1[2] : 1.f - l1[2]);
          const long long p = (((long long)b * D + (dz ? i1[0] : i0[0])) * H + (dy ? i1[1] : i0[1])) * W + (dx ? i1[2] : i0[2]);
          const uint4 q = __ldg(reinterpret_cast<const uint4*>(in + p * in_ctot + in_coff + ch));
          const T* e = reinterpret_cast<const T*>(&q);
#pragma unroll
          for (int k = 0; k < VEC; ++k) acc[k] = fmaf(wgt, (float)e[k], acc[k]);
        }
    uint4 q;
    T* e = reinterpret_cast<T*>(&q);
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      float v = acc[k];
      if (sizeof(T) == 4 && round_tf32) { uint32_t u; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v)); v = __uint_as_float(u); }
      e[k] = (T)v;
    }
    const long long op = (((long long)b * oD + z) * oH + y) * oW + x;
    *reinterpret_cast<uint4*>(out + op * out_ctot + out_coff + ch) = q;
  }
}

// Bilinear x2 up-sampling with align_corners=True (nn.Upsample in multi_output_nested_unet.py:74): source coordinate
// o * (n - 1) / (2n - 1) in float32, the four neighbours combined in PyTorch's order
// h0 * (w0 * v00 + w1 * v01) + h1 * (w0 * v10 + w1 * v11); NHWC, 16-byte channel vectors.
// Output rows 2p-1 and 2p (columns 2q-1 and 2q) interpolate between the SAME two source rows (columns) p-1 and p, so a
// thread loads one 2 x 2 source neighbourhood and produces the 2 x 2 output block: a quarter of the loads and half
// of the arithmetic of a per-output-pixel kernel. The coordinates of every output row / column are still computed
// with PyTorch's expression; should they ever disagree inside a pair, the pixel takes the generic path.
__device__ __forceinline__ void bilinear_coord(int o, float s, int n, int& i0, int& i1, float& l1) {
  const float f = s * (float)o;
  i0 = min((int)f, n - 1);
  i1 = min(i0 + 1, n - 1);
  l1 = fminf(fmaxf(f - (float)i0, 0.f), 1.f);
}
template <typename T, int VEC>
__device__ __forceinline__ void bilinear_load(const T* p, float (&f)[VEC]) {
  const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
  const T* e = reinterpret_cast<const T*>(&q);
#pragma unroll
  for (int k = 0; k < VEC; ++k) f[k] = (float)e[k];
}
template <typename T, int VEC>
__device__ __forceinline__ void bilinear_store(T* p, const float (&t)[VEC], const float (&bt)[VEC], float h0, float h1,
                                               int round_tf32) {
  uint4 q;
  T* e = reinterpret_cast<T*>(&q);
#pragma unroll
  for (int k = 0; k < VEC; ++k) {
    float v = h0 * t[k] + h1 * bt[k];
    if (sizeof(T) == 4 && round_tf32) { uint32_t u; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v)); v = __uint_as_float(u); }
    e[k] = (T)v;
  }
  *reinterpret_cast<uint4*>(p) = q;
}

template <typename T, int VEC>
__global__ void __launch_bounds__(256) up_bilinear_kernel(const T* __restrict__ in, int in_ctot, int in_coff, int c,
                                                          int B, int H, int W, T* __restrict__ out, int out_ctot,
                                                          int out_coff, int round_tf32) {
  const int oH = 2 * H, oW = 2 * W, cv = c / VEC;
  const float sh = (float)(H - 1) / (float)(oH - 1), sw = (float)(W - 1) / (float)(oW - 1);
  const int items = B * (H + 1), per_item = (W + 1) * cv;
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    const int b = item / (H + 1), p = item - b * (H + 1);
    const bool va = p >= 1, vb = p < H;                 // output rows 2p-1 / 2p exist
    const int ya = va ? 2 * p - 1 : 2 * p, yb = vb ? 2 * p : 2 * p - 1;
    int ya0, ya1, yb0, yb1;
    float ha1, hb1;
    bilinear_coord(ya, sh, H, ya0, ya1, ha1);
    bilinear_coord(yb, sh, H, yb0, yb1, hb1);
    const bool rows_shared = ya0 == yb0 && ya1 == yb1;
    const T* img = in + (long long)b * H * W * in_ctot + in_coff;
    T* oimg = out + (long long)b * oH * oW * out_ctot + out_coff;
    for (int i = threadIdx.x; i < per_item; i += blockDim.x) {
      const int q = i / cv, chn = (i - q * cv) * VEC;
      const bool ua = q >= 1, ub = q < W;
      const int xa = ua ? 2 * q - 1 : 2 * q, xb = ub ? 2 * q : 2 * q - 1;
      int xa0, xa1, xb0, xb1;
      float wa1, wb1;
      bilinear_coord(xa, sw, W, xa0, xa1, wa1);
      bilinear_coord(xb, sw, W, xb0, xb1, wb1);
      if (rows_shared && xa0 == xb0 && xa1 == xb1) {
        float v00[VEC], v01[VEC], v10[VEC], v11[VEC];
        bilinear_load<T, VEC>(img + ((long long)ya0 * W + xa0) * in_ctot + chn, v00);
        bilinear_load<T, VEC>(img + ((long long)ya0 * W + xa1) * in_ctot + chn, v01);
        bilinear_load<T, VEC>(img + ((long long)ya1 * W + xa0) * in_ctot + chn, v10);
        bilinear_load<T, VEC>(img + ((long long)ya1 * W + xa1) * in_ctot + chn, v11);
        float ta[VEC], tb[VEC], ba[VEC], bb[VEC];       // horizontal lerps of the top / bottom source row at xa / xb
        const float wa0 = 1.f - wa1, wb0 = 1.f - wb1;
#pragma unroll
        for (int k = 0; k < VEC; ++k) {
          ta[k] = wa0 * v00[k] + wa1 * v01[k];
          tb[k] = wb0 * v00[k] + wb1 * v01[k];
          ba[k] = wa0 * v10[k] + wa1 * v11[k];
          bb[k] = wb0 * v10[k] + wb1 * v11[k];
        }
        if (va) {
          T* orow = oimg + (long long)(2 * p - 1) * oW * out_ctot + chn;
          if (ua) bilinear_store<T, VEC>(orow + (long long)(2 * q - 1) * out_ctot, ta, ba, 1.f - ha1, ha1, round_tf32);
          if (ub) bilinear_store<T, VEC>(orow + (long long)(2 * q) * out_ctot, tb, bb, 1.f - ha1, ha1, round_tf32);
        }
        if (vb) {
          T* orow = oimg + (long long)(2 * p) * oW * out_ctot + chn;
          if (ua) bilinear_store<T, VEC>(orow + (long long)(2 * q - 1) * out_ctot, ta, ba, 1.f - hb1, hb1, round_tf32);
          if (ub) bilinear_store<T, VEC>(orow + (long long)(2 * q) * out_ctot, tb, bb, 1.f - hb1, hb1, round_tf32);
        }
      } else {
        // generic path, one output pixel at a time (never taken for the extents this engine plans)
        for (int r = 0; r < 2; ++r) {
          if (!(r ? vb : va)) continue;
          const int y = 2 * p - 1 + r;
          int y0, y1; float h1;
          bilinear_coord(y, sh, H, y0, y1, h1);
          for (int cidx = 0; cidx < 2; ++cidx) {
            if (!(cidx ? ub : ua)) continue;
            const int x = 2 * q - 1 + cidx;
            int x0, x1; float w1;
            bilinear_coord(x, sw, W, x0, x1, w1);
            float v00[VEC], v01[VEC], v10[VEC], v11[VEC], t[VEC], bt[VEC];
            bilinear_load<T, VEC>(img + ((long long)y0 * W + x0) * in_ctot + chn, v00);
            bilinear_load<T, VEC>(img + ((long long)y0 * W + x1) * in_ctot + chn, v01);
            bilinear_load<T, VEC>(img + ((long long)y1 * W + x0) * in_ctot + chn, v10);
            bilinear_load<T, VEC>(img + ((long long)y1 * W + x1) * in_ctot + chn, v11);
#pragma unroll
            for (int k = 0; k < VEC; ++k) {
              t[k] = (1.f - w1) * v00[k] + w1 * v01[k];
              bt[k] = (1.f - w1) * v10[k] + w1 * v11[k];
            }
            bilinear_store<T, VEC>(oimg + ((long long)y * oW + x) * out_ctot + chn, t, bt, 1.f - h1, h1, round_tf32);
          }
        }
      }
    }
  }
}

// skip[pix][c] *= psi[pix] on one half of a concat buffer (AttentionBlock: out = skip_connection * psi)
template <int FMT>
__global__ void mul_psi_kernel(void* act, int ctot, int coff, int c, const float* __restrict__ psi, long long npix,
                               int round_tf32) {
  constexpr int esz = fmt_esz(FMT);
  const int vec = 16 / esz, cv = c / vec;
  const long long total = npix * cv;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pix = i / cv;
    const int v = (int)(i - pix * cv);
    const float s = __ldg(psi + pix);
    uint4* ptr = reinterpret_cast<uint4*>(reinterpret_cast<char*>(act) + ((pix * ctot + coff) * esz + (long long)v * 16));
    uint4 x = *ptr;
    if (FMT == FMT_F16) {
      __half2* xp = reinterpret_cast<__half2*>(&x);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float2 f = __half22float2(xp[k]);
        xp[k] = __floats2half2_rn(f.x * s, f.y * s);
      }
    } else if (esz == 2) {
      __nv_bfloat162* xp = reinterpret_cast<__nv_bfloat162*>(&x);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float2 f = __bfloat1622float2(xp[k]);
        xp[k] = __floats2bfloat162_rn(f.x * s, f.y * s);
      }
    } else {
      float* xp = reinterpret_cast<float*>(&x);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float t = xp[k] * s;
        if (round_tf32) { uint32_t u; asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(t)); t = __uint_as_float(u); }
        xp[k] = t;
      }
    }
    *ptr = x;
  }
}

int net_forward(Net* n, const void* in, int in_kind, const void* in2, float* out_val, uint8_t* out_u8,
                void* workspace, cudaStream_t stream) {
  BIU_REQUIRE(n->finalized, "network weights were not finalized");
  BIU_REQUIRE(n->B > 0, "biu_net_plan must be called before biu_net_forward");
  char* ws = reinterpret_cast<char*>(workspace);
  const bool tc_allowed = n->fmt != FMT_F32 && !n->force_direct;
  const int esz = fmt_esz(n->fmt);
  const int round_tf32 = n->fmt == FMT_TF32 ? 1 : 0;   // flag of the join and up-sampling kernels below
  if (n->profile && n->events.size() < 2 * n->ops.size()) {
    while (n->events.size() < 2 * n->ops.size()) {
      cudaEvent_t e;
      BIU_CHECK_CUDA(cudaEventCreate(&e));
      n->events.push_back(e);
    }
  }
  n->op_kinds.assign(n->ops.size(), 0);
  n->stopped = false;
  int op_index = -1;
  bool skip_pool = false;           // the previous convolution wrote the pooled tensor from its epilogue
  for (const Op& o : n->ops) {
    ++op_index;
    // debug stop: the ops up to debug_stop ran exactly as in a full forward (fusion included: a pool fused into
    // op debug_stop's epilogue has been written); nothing after it runs, so a test can read what op debug_stop wrote
    // before a later op reuses the buffer
    if (n->debug_stop >= 0 && op_index > n->debug_stop) { n->stopped = true; break; }
    if (n->profile && op_index > 0) BIU_CHECK_CUDA(cudaEventRecord(n->events[2 * op_index - 1], stream));
    if (n->profile) BIU_CHECK_CUDA(cudaEventRecord(n->events[2 * op_index], stream));
    n->op_kinds[op_index] = (int)o.kind;
    if (skip_pool && o.kind == OP_POOL) { skip_pool = false; n->op_kinds[op_index] += 32; continue; }
    skip_pool = false;
    int d, h, w;
    level_dims(n, o.level, &d, &h, &w);
    // twin-encoder buffers hold two image streams: [current (B) | previous (B)], or with the shared encoder the unique
    // tiles, previous stream = images [0, B) and current stream = images [shared, shared + B)
    const int shared = (n->kind == NET_SIAM2D && n->siam_mode != SIAM_CONTROL) ? n->siam_shared : 0;
    auto stream_img0 = [&](const Buf* bf, int stream) -> size_t {
      if (bf->batch_mul == 2 && shared > 0) return stream == 0 ? (size_t)shared : 0;
      return (size_t)stream * n->B;
    };
    const int batch = (o.batch_mul == 2 && shared > 0) ? n->B + shared : n->B * o.batch_mul;
    const Buf* sb = o.src >= 0 ? &n->bufs[o.src] : nullptr;
    const Buf* db = o.dst >= 0 ? &n->bufs[o.dst] : nullptr;
    const size_t img_in = sb ? (size_t)d * h * w * sb->ctot * esz : 0;
    // an op that covers both streams (batch_mul 2) starts at image 0 of the buffer
    const char* src = sb ? ws + sb->offset + (o.batch_mul == 2 ? 0 : stream_img0(sb, o.src_img0)) * img_in : nullptr;
    auto dst_ptr = [&](int dd, int hh, int ww) -> char* {
      return db ? ws + db->offset + (o.batch_mul == 2 ? 0 : stream_img0(db, o.dst_img0)) *
                                        ((size_t)dd * hh * ww * db->ctot * esz) : nullptr;
    };
    switch (o.kind) {
      case OP_FIRST: {
        const ConvLayer& L = n->layers[o.layer];
        FirstConvArgs a;
        memset(&a, 0, sizeof(a));
        a.in_kind = in_kind;
        a.in = o.src == -1 ? in : in2;
        if (shared > 0) {                    // one pass over the B + shared unique tiles, given as ONE array
          if (o.src != -1) { n->op_kinds[op_index] += 32; break; }
          BIU_REQUIRE(in2 == nullptr, "shared twin encoder: the unique tiles come as one array (no second input)");
        }
        BIU_REQUIRE(a.in != nullptr, "network input pointer is null");
        a.cin = n->in_ch; a.W = w; a.H = h; a.D = d; a.B = shared > 0 ? n->B + shared : n->B; a.kd = L.kd;
        a.wgt = L.w_direct; a.cout = L.cout_pad; a.cout_real = L.cout; a.slope = L.slope; a.scale = L.scale; a.shift = L.shift;
        a.fmt = n->fmt; a.out = shared > 0 ? ws + db->offset : dst_ptr(d, h, w); a.out_ctot = db->ctot; a.out_coff = o.dst_coff;
        a.cout_pad = L.cout_pad;
        if (tc_allowed && in_kind == 0 && n->dims == 2 && a.D == 1 && L.w_first != nullptr) {
          FirstRowsArgs fr;
          memset(&fr, 0, sizeof(fr));
          fr.fmt = n->fmt; fr.in = reinterpret_cast<const uint8_t*>(a.in); fr.W = a.W; fr.H = a.H; fr.B = a.B;
          fr.wgt = L.w_first; fr.n_total = L.cout_pad; fr.slope = L.slope; fr.scale = L.scale_first; fr.shift = L.shift;
          fr.out = a.out; fr.out_ctot = a.out_ctot; fr.out_coff = a.out_coff;
          if (conv_first_rows_supported(fr)) {
            if (int rc = launch_conv_first_rows(fr, stream)) return rc;
            break;
          }
        }
        if (int rc = launch_first_conv(a, stream)) return rc;
        break;
      }
      case OP_CONV:
      case OP_CONV_HEAD: {
        const ConvLayer& L = n->layers[o.layer];
        const bool head = o.kind == OP_CONV_HEAD;
        ConvTcArgs a;
        memset(&a, 0, sizeof(a));
        a.fmt = n->fmt; a.in = src; a.in_ctot = sb->ctot; a.in_coff = o.src_coff; a.cin = L.cin_phys;
        a.W = w; a.H = h; a.D = d; a.B = batch; a.kw = L.kw; a.kh = L.kh; a.kd = L.kd;
        a.wgt = L.w_tc; a.wgt_fold = L.w_fold; a.wgt_fold_z = L.w_fold_z; a.n_total = L.cout_pad; a.mode = head ? EPI_HEAD : EPI_CONV; a.slope = L.slope;
        a.scale = L.scale; a.shift = L.shift;
        a.out = head ? nullptr : dst_ptr(d, h, w);
        a.out_ctot = head ? 0 : db->ctot; a.out_coff = o.dst_coff;
        if (n->acc_scratch >= 0 && o.level > 0 && o.src != n->acc_scratch && o.dst != n->acc_scratch) {
          const Buf& sc = n->bufs[n->acc_scratch];     // level-0 buffer: dead once the encoder has left level 0
          int d0, h0, w0;
          level_dims(n, sc.level, &d0, &h0, &w0);
          a.acc_scratch = ws + sc.offset;
          a.acc_scratch_bytes = (long long)n->B * sc.batch_mul * d0 * h0 * w0 * sc.ctot * esz;
        }
        if (head) {
          a.head_n = n->head_total; a.head_w = n->head_w; a.head_b = n->head_b;
          int row = 0;
          for (size_t hi = 0; hi < n->head_channels.size(); ++hi)
            for (int c = 0; c < n->head_channels[hi]; ++c) a.head_act[row++] = n->head_acts[hi];
          a.out_val = out_val; a.out_u8 = out_u8;
        }
        if (tc_allowed && L.w_tc && conv_tc_supported(a)) {
          // MaxPool2d(2) directly after this block (unet/unet.py:73-74 etc.): fused into the epilogue
          if (!head && n->dims == 2 && !n->no_fuse && op_index + 1 < (int)n->ops.size()) {
            const Op& nx = n->ops[op_index + 1];
            if (nx.kind == OP_POOL && nx.pool_mode == 0 && nx.src == o.dst && nx.src_coff == o.dst_coff &&
                nx.c == L.cout_pad && nx.batch_mul == o.batch_mul && nx.src_img0 == 0 && nx.dst_img0 == 0 &&
                o.dst_img0 == 0 && nx.level == o.level) {
              const Buf& pb = n->bufs[nx.dst];
              a.pool_out = ws + pb.offset; a.pool_ctot = pb.ctot; a.pool_coff = nx.dst_coff;
              if (conv_tc_can_fuse_pool(a)) skip_pool = true;
              else a.pool_out = nullptr;
            }
          }
          // MaxPool3d(2) after a full-resolution block (unet3d/unet3d.py:66-73): the row kernel's epilogue pools every
          // plane in (y, x) into an idle decoder buffer, a second pass over a quarter of the data reduces the z pairs
          bool zpairs = false;
          PoolArgs zp;
          // first choice, any level: the row kernel's plane mode streams the planes of a tile in pairs and pools in
          // (z, y, x) straight into the pool's destination
          if (!head && n->dims == 3 && !n->no_fuse && op_index + 1 < (int)n->ops.size()) {
            const Op& nx = n->ops[op_index + 1];
            if (nx.kind == OP_POOL && nx.pool_mode == 0 && nx.src == o.dst && nx.src_coff == o.dst_coff &&
                nx.c == L.cout_pad && nx.batch_mul == 1 && o.batch_mul == 1 && nx.level == o.level &&
                nx.src_img0 == 0 && nx.dst_img0 == 0 && o.dst_img0 == 0) {
              const Buf& pb = n->bufs[nx.dst];
              a.pool_out = ws + pb.offset; a.pool_ctot = pb.ctot; a.pool_coff = nx.dst_coff; a.pool_3d = 1;
              if (conv_tc_can_fuse_pool3d(a)) skip_pool = true;
              else { a.pool_out = nullptr; a.pool_3d = 0; }
            }
          }
          if (!skip_pool && !head && n->dims == 3 && !n->no_fuse && o.level == 0 && n->pool_scratch >= 0 &&
              op_index + 1 < (int)n->ops.size()) {
            const Op& nx = n->ops[op_index + 1];
            if (nx.kind == OP_POOL && nx.pool_mode == 0 && nx.src == o.dst && nx.src_coff == o.dst_coff &&
                nx.c == L.cout_pad && nx.batch_mul == 1 && o.batch_mul == 1 && nx.level == 0) {
              const Buf& sc = n->bufs[n->pool_scratch];
              const Buf& pb = n->bufs[nx.dst];
              a.pool_out = ws + sc.offset; a.pool_ctot = L.cout_pad; a.pool_coff = 0;
              if (conv_tc_can_fuse_pool_xy(a)) {
                zpairs = skip_pool = true;
                memset(&zp, 0, sizeof(zp));
                zp.fmt = n->fmt; zp.in = a.pool_out; zp.in_ctot = L.cout_pad; zp.in_coff = 0; zp.c = L.cout_pad;
                zp.W = w / 2; zp.H = h / 2; zp.D = d; zp.B = batch; zp.dims = 3; zp.mode = 2;
                zp.out = ws + pb.offset; zp.out_ctot = pb.ctot; zp.out_coff = nx.dst_coff;
              } else {
                a.pool_out = nullptr;
              }
            }
          }
          if (int rc = launch_conv_tc(a, stream)) return rc;
          if (zpairs) { if (int rc = launch_pool2(zp, stream)) return rc; }
        } else {
          n->op_kinds[op_index] += 16;
          DirectConvArgs da;
          memset(&da, 0, sizeof(da));
          da.fmt = n->fmt; da.in = src; da.in_ctot = sb->ctot; da.in_coff = o.src_coff; da.cin = L.cin_phys;
          da.W = w; da.H = h; da.D = d; da.B = batch; da.kw = L.kw; da.kh = L.kh; da.kd = L.kd;
          da.wgt = L.w_direct; da.cout = L.cout_pad; da.slope = L.slope; da.scale = L.scale; da.shift = L.shift;
          if (!head) {
            da.out = dst_ptr(d, h, w); da.out_ctot = db->ctot; da.out_coff = o.dst_coff;
            if (int rc = launch_direct_conv(da, stream)) return rc;
          } else {
            // reuse the (now dead) first encoder buffer of level 0 as scratch for the last activation
            const Buf& scratch = n->bufs[0];
            BIU_REQUIRE(scratch.level == 0 && scratch.ctot >= L.cout_pad, "no scratch buffer for the head");
            da.out = ws + scratch.offset; da.out_ctot = scratch.ctot; da.out_coff = 0;
            if (int rc = launch_direct_conv(da, stream)) return rc;
            HeadArgs ha;
            memset(&ha, 0, sizeof(ha));
            ha.fmt = n->fmt; ha.in = da.out; ha.in_ctot = scratch.ctot; ha.in_coff = 0; ha.cin = L.cout_pad;
            ha.npix_per_img = (long long)d * h * w; ha.B = batch; ha.head_n = n->head_total;
            ha.w = n->head_w; ha.b = n->head_b;
            int row = 0;
            for (size_t hi = 0; hi < n->head_channels.size(); ++hi)
              for (int c = 0; c < n->head_channels[hi]; ++c) ha.act[row++] = n->head_acts[hi];
            ha.out_val = out_val; ha.out_u8 = out_u8;
            if (int rc = launch_head(ha, stream)) return rc;
          }
        }
        break;
      }
      case OP_UP: {
        const ConvLayer& L = n->layers[o.layer];
        const int od = n->dims == 3 ? 2 * d : d;
        ConvTcArgs a;
        memset(&a, 0, sizeof(a));
        a.fmt = n->fmt; a.in = src; a.in_ctot = sb->ctot; a.in_coff = o.src_coff; a.cin = L.cin_phys;
        a.W = w; a.H = h; a.D = d; a.B = batch; a.kw = a.kh = a.kd = 1;
        a.wgt = L.w_tc; a.n_total = L.nq * L.cout_pad; a.mode = EPI_UP; a.slope = 1.f;
        a.scale = L.scale; a.shift = L.shift;
        a.out = dst_ptr(od, 2 * h, 2 * w); a.out_ctot = db->ctot; a.out_coff = o.dst_coff;
        a.up_cout = L.cout_pad; a.up_dims = n->dims;
        if (tc_allowed && L.w_tc && conv_tc_supported(a)) {
          if (int rc = launch_conv_tc(a, stream)) return rc;
        } else {
          n->op_kinds[op_index] += 16;
          DirectUpArgs da;
          memset(&da, 0, sizeof(da));
          da.fmt = n->fmt; da.in = src; da.in_ctot = sb->ctot; da.in_coff = o.src_coff; da.cin = L.cin_phys;
          da.W = w; da.H = h; da.D = d; da.B = batch; da.dims = n->dims; da.wgt = L.w_direct; da.bias = L.shift;
          da.cout = L.cout_pad; da.out = a.out; da.out_ctot = db->ctot; da.out_coff = o.dst_coff;
          if (int rc = launch_direct_up(da, stream)) return rc;
        }
        break;
      }
      case OP_POOL: {
        PoolArgs a;
        memset(&a, 0, sizeof(a));
        a.fmt = n->fmt; a.in = src; a.in_ctot = sb->ctot; a.in_coff = o.src_coff; a.c = o.c;
        a.W = w; a.H = h; a.D = d; a.B = batch; a.dims = n->dims; a.mode = o.pool_mode;
        a.out = dst_ptr(n->dims == 3 ? d / 2 : d, h / 2, w / 2); a.out_ctot = db->ctot; a.out_coff = o.dst_coff;
        if (int rc = launch_pool2(a, stream)) return rc;
        break;
      }
      case OP_UPNEAREST: {
        UpNearestArgs a;
        memset(&a, 0, sizeof(a));
        a.fmt = n->fmt; a.in = src; a.in_ctot = sb->ctot; a.in_coff = o.src_coff; a.c = o.c;
        a.W = w; a.H = h; a.D = d; a.B = batch; a.dims = n->dims;
        a.out = dst_ptr(n->dims == 3 ? 2 * d : d, 2 * h, 2 * w); a.out_ctot = db->ctot; a.out_coff = o.dst_coff;
        if (int rc = launch_up_nearest(a, stream)) return rc;
        break;
      }
      case OP_GATE: {
        const ConvLayer& L = n->layers[o.layer];
        float* psi = reinterpret_cast<float*>(ws + db->offset);
        ConvTcArgs a;
        memset(&a, 0, sizeof(a));
        a.fmt = n->fmt; a.in = src; a.in_ctot = sb->ctot; a.in_coff = o.src_coff; a.cin = L.cin_phys;
        a.W = w; a.H = h; a.D = d; a.B = batch; a.kw = a.kh = a.kd = 1;
        a.wgt = L.w_tc; a.n_total = L.cout_pad; a.mode = EPI_HEAD; a.slope = 0.f;
        a.scale = L.scale; a.shift = L.shift; a.out = nullptr;
        a.head_n = 1; a.head_w = L.gate_w; a.head_b = L.gate_b; a.head_act[0] = ACT_SIGMOID;
        a.out_val = psi; a.out_u8 = nullptr;
        if (tc_allowed && L.w_tc && conv_tc_supported(a)) {
          if (int rc = launch_conv_tc(a, stream)) return rc;
        } else {
          n->op_kinds[op_index] += 16;
          BIU_REQUIRE(n->gate_scratch >= 0, "no scratch buffer for the attention gate");
          const Buf& scratch = n->bufs[n->gate_scratch];
          DirectConvArgs da;
          memset(&da, 0, sizeof(da));
          // the gate's activation only feeds psi below and is read by no tensor-core kernel: fp32 stays unrounded
          da.fmt = n->fmt == FMT_TF32 ? FMT_F32 : n->fmt;
          da.in = src; da.in_ctot = sb->ctot; da.in_coff = o.src_coff; da.cin = L.cin_phys;
          da.W = w; da.H = h; da.D = d; da.B = batch; da.kw = da.kh = da.kd = 1;
          da.wgt = L.w_direct; da.cout = L.cout_pad; da.slope = 0.f; da.scale = L.scale; da.shift = L.shift;
          da.out = ws + scratch.offset; da.out_ctot = L.cout_pad; da.out_coff = 0;
          if (int rc = launch_direct_conv(da, stream)) return rc;
          HeadArgs ha;
          memset(&ha, 0, sizeof(ha));
          ha.fmt = da.fmt; ha.in = da.out; ha.in_ctot = L.cout_pad; ha.in_coff = 0; ha.cin = L.cout_pad;
          ha.npix_per_img = (long long)d * h * w; ha.B = batch; ha.head_n = 1;
          ha.w = L.gate_w; ha.b = L.gate_b; ha.act[0] = ACT_SIGMOID;
          ha.out_val = psi; ha.out_u8 = nullptr;
          if (int rc = launch_head(ha, stream)) return rc;
        }
        break;
      }
      case OP_MULPSI: {
        const long long npix = (long long)batch * d * h * w;
        const int vec = 16 / esz;
        long long blocks = ceil_div_ll(npix * (o.c / vec), 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        if (blocks < 1) blocks = 1;
        float* psi = reinterpret_cast<float*>(ws + sb->offset);
        if (int rc = with_elem_type(n->fmt, [&](auto tag) {
              mul_psi_kernel<decltype(tag)::fmt><<<(int)blocks, 256, 0, stream>>>(
                  ws + db->offset, db->ctot, o.dst_coff, o.c, psi, npix, round_tf32);
              return 0;
            }))
          return rc;
        BIU_CHECK_CUDA(cudaGetLastError());
        count_launch();
        break;
      }
      case OP_XCORR: {
        const size_t img = (size_t)d * h * w * sb->ctot * esz;
        int G = 8;
        while (G > 1 && (size_t)2 * h * w * G * sizeof(float) > 96 * 1024) G >>= 1;
        const size_t smem = (size_t)2 * h * w * G * sizeof(float);
        BIU_REQUIRE(smem <= 200 * 1024, "Siam_UNet mode='corr': a %dx%d embedding does not fit shared memory", h, w);
        const int blocks = n->B * (sb->ctot / G);
        const char* cur = ws + sb->offset + img * stream_img0(sb, 0);
        const char* prv = ws + sb->offset + img * stream_img0(sb, 1);
        if (int rc = with_elem_type(n->fmt, [&](auto tag) {
              using T = typename decltype(tag)::type;
              if (smem > 48 * 1024)
                BIU_CHECK_CUDA(cudaFuncSetAttribute(xcorr_join_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
              xcorr_join_kernel<T><<<blocks, 256, smem, stream>>>(reinterpret_cast<const T*>(cur), reinterpret_cast<const T*>(prv),
                                                                   reinterpret_cast<T*>(ws + db->offset), h, w, sb->ctot, G,
                                                                   round_tf32);
              return 0;
            }))
          return rc;
        BIU_CHECK_CUDA(cudaGetLastError());
        count_launch();
        break;
      }
      case OP_UPTRILINEAR: {
        const long long total = (long long)batch * 8 * d * h * w * (o.c / (16 / esz));
        long long blocks = ceil_div_ll(total, 256);
        if (blocks > 148 * 16) blocks = 148 * 16;
        if (blocks < 1) blocks = 1;
        char* dst = ws + db->offset;
        if (int rc = with_elem_type(n->fmt, [&](auto tag) {
              using T = typename decltype(tag)::type;
              up_trilinear_kernel<T, 16 / sizeof(T)><<<(int)blocks, 256, 0, stream>>>(
                  reinterpret_cast<const T*>(src), sb->ctot, o.src_coff, o.c, batch, d, h, w, reinterpret_cast<T*>(dst), db->ctot,
                  o.dst_coff, round_tf32);
              return 0;
            }))
          return rc;
        BIU_CHECK_CUDA(cudaGetLastError());
        count_launch();
        break;
      }
      case OP_UPBILINEAR: {
        int blocks = batch * (h + 1);                      // one block iteration per pair of output rows
        if (blocks > 148 * 8) blocks = 148 * 8;
        char* dst = ws + db->offset;
        if (int rc = with_elem_type(n->fmt, [&](auto tag) {
              using T = typename decltype(tag)::type;
              up_bilinear_kernel<T, 16 / sizeof(T)><<<blocks, 256, 0, stream>>>(
                  reinterpret_cast<const T*>(src), sb->ctot, o.src_coff, o.c, batch, h, w, reinterpret_cast<T*>(dst), db->ctot,
                  o.dst_coff, round_tf32);
              return 0;
            }))
          return rc;
        BIU_CHECK_CUDA(cudaGetLastError());
        count_launch();
        break;
      }
      case OP_MAXJOIN: {
        const size_t img = (size_t)d * h * w * sb->ctot * esz;
        const long long nvec = (long long)(img * n->B / 16);
        long long blocks = ceil_div_ll(nvec, 256);
        if (blocks > 148 * 8) blocks = 148 * 8;
        if (blocks < 1) blocks = 1;
        const uint4* xa = reinterpret_cast<const uint4*>(ws + sb->offset + img * stream_img0(sb, 0));
        const uint4* xb = reinterpret_cast<const uint4*>(ws + sb->offset + img * stream_img0(sb, 1));
        uint4* xo = reinterpret_cast<uint4*>(ws + db->offset);
        if (int rc = with_elem_type(n->fmt, [&](auto tag) {
              max_join_kernel<decltype(tag)::fmt><<<(int)blocks, 256, 0, stream>>>(xa, xb, xo, nvec);
              return 0;
            }))
          return rc;
        BIU_CHECK_CUDA(cudaGetLastError());
        count_launch();
        break;
      }
    }
  }
  if (n->profile && !n->ops.empty() && !n->stopped)
    BIU_CHECK_CUDA(cudaEventRecord(n->events[2 * n->ops.size() - 1], stream));
  return 0;
}

int net_profile_read(Net* n, int max_ops, int* kinds, float* ms, int* n_ops) {
  BIU_REQUIRE(n->profile && n->events.size() >= 2 * n->ops.size(), "profiling was not enabled for the last forward");
  BIU_REQUIRE(!n->stopped, "the last forward stopped after op %d (biu_net_set_debug_stop): the later ops have no "
              "timings", n->debug_stop);
  const int cnt = (int)n->ops.size() < max_ops ? (int)n->ops.size() : max_ops;
  for (int i = 0; i < cnt; ++i) {
    BIU_CHECK_CUDA(cudaEventSynchronize(n->events[2 * i + 1]));
    BIU_CHECK_CUDA(cudaEventElapsedTime(&ms[i], n->events[2 * i], n->events[2 * i + 1]));
    kinds[i] = n->op_kinds[i];
  }
  *n_ops = cnt;
  return 0;
}

int net_debug_copy(Net* n, const char* buf_name, void* workspace, void* dst_host, long long max_bytes) {
  for (auto& b : n->bufs) {
    if (b.name == buf_name) {
      int d, h, w;
      level_dims(n, b.level, &d, &h, &w);
      const long long imgs = (b.batch_mul == 2 && n->siam_shared > 0) ? (long long)n->B + n->siam_shared : (long long)n->B * b.batch_mul;
      long long bytes = imgs * d * h * w * b.ctot * fmt_esz(n->fmt);
      if (bytes > max_bytes) bytes = max_bytes;
      BIU_CHECK_CUDA(cudaMemcpy(dst_host, reinterpret_cast<char*>(workspace) + b.offset, bytes, cudaMemcpyDeviceToHost));
      return 0;
    }
  }
  BIU_REQUIRE(false, "no activation buffer named '%s'", buf_name);
}

void net_destroy(Net* n) {
  for (void* p : n->dev_allocs) cudaFree(p);
  for (cudaEvent_t e : n->events) cudaEventDestroy(e);
  delete n;
}

}  // namespace biu
