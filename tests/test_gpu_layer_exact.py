"""Every op of the layer program against an exact single-op reference (tests/_layer_ref.py).

Each case plans a network, runs one profiled forward and recomputes every op of the program from the engine's OWN
stored input, in float64: convolutions and transposed convolutions must give the correctly rounded value (up to the
fp32 accumulation allowance), pools, nearest up-sampling and the Siam max join the exact maximum / copy, trilinear and
bilinear up-sampling, the Siam cross-correlation and the attention gate their interval, mul_psi the rounded product,
heads act(sum h_w v + h_b) within 1e-5. Ops whose input and output survive the forward are checked from it; every
other op k is checked after a forward that stops after op k (Engine.set_debug_stop), so no op is skipped. Nothing
compounds through the network, so a single wrong tap, rounding mode or scale index in any kernel variant fails here.

The program below mirrors net_build (bio_image_unet_b200/csrc/net.cu) for every network kind; the length and op
kinds of the engine's profile must match it, so a change of the program fails loudly. The other families' cases are
in tests/test_gpu_layer_exact_families.py.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests import _layer_ref as R

pytestmark = pytest.mark.gpu

FIRST, CONV, HEAD, UP, POOL, UPNEAREST, MAXJOIN, GATE, MULPSI, XCORR, UPTRI, UPBILINEAR = range(12)
pad16 = R.pad16
HEAD_ACT = {'': 'sigmoid'}
KINDS_2D = ('unet2d', 'attunet2d', 'siam2d', 'unet2d_v0', 'mo2d', 'nested2d', 'nested2d_3l')


# ------------------------------------------------------------------------------------------------ program mirror
def _op(kind, layer, src, src_coff, dst, dst_coff, c, level, segs=None, cout=None, pool_mode=0, bm=1, src_img0=0,
        dst_img0=0, keys=None):
    """keys: state_dict prefixes (conv, BatchNorm) of the layer, '<layer>.0' / '<layer>.1' by default. bm: the op runs
    on both image streams of a twin-encoder buffer; src_img0 / dst_img0: the stream of a one-stream op."""
    if keys is None and layer is not None:
        keys = (layer + '.0', layer + '.1')
    return dict(kind=kind, layer=layer, src=src, src_coff=src_coff, dst=dst, dst_coff=dst_coff, c=c, level=level,
                segs=segs or [(0, c, 0)], cout=cout, pool_mode=pool_mode, bm=bm, src_img0=src_img0, dst_img0=dst_img0,
                keys=keys)


def _program_unet2d(kind, nf, siam_mode):
    """Unet / AttentionUnet / Siam_UNet / Unet_v0 / MultiOutputUnet: the first branch of net_build."""
    bufs, ops = {}, []
    siam, v0, att = kind == 'siam2d', kind == 'unet2d_v0', kind == 'attunet2d'
    bm = 2 if siam and siam_mode != 'control' else 1
    ch = [nf << i for i in range(5)]
    for l in range(4):
        bufs[f'e{2 * l + 1}'] = (l, pad16(ch[l]), bm)
        bufs[f'cat{4 - l}'] = (l, 2 * pad16(ch[l]), bm)
        bufs[f'm{l + 1}'] = (l + 1, pad16(ch[l]), bm)
    if siam and siam_mode == 'concat':
        bufs['joincat'] = (4, 2 * pad16(ch[3]), 1)
    if siam and siam_mode != 'control':
        bufs['join'] = (4, pad16(ch[3]), 1)
    bufs['mid1'] = bufs['mid2'] = (4, pad16(ch[4]), 1)
    da, db = {}, {}
    for l in range(3, -1, -1):
        da[l] = f'd{2 * (3 - l) + 1}'
        bufs[da[l]] = (l, pad16(ch[l]), 1)
        if l > 0 or v0:
            db[l] = f'd{2 * (3 - l) + 2}'
            bufs[db[l]] = (l, pad16(ch[l]), 1)
        if att:
            bufs[f'psi{4 - l}'] = (l, None, 1)
    for l in range(4):
        e, cat, p = f'e{2 * l + 1}', f'cat{4 - l}', pad16(ch[l])
        # the skip lives in the upper half of the concat buffer: the second conv's output, Unet_v0's first
        c1_dst, c1_coff = (cat, p) if v0 else (e, 0)
        if l == 0:
            ops.append(_op(FIRST, 'encode1', None, 0, c1_dst, c1_coff, 1, 0, cout=ch[0]))
            if bm == 2:
                ops.append(_op(FIRST, 'encode1', None, 0, c1_dst, c1_coff, 1, 0, cout=ch[0], src_img0=1, dst_img0=1))
        else:
            ops.append(_op(CONV, f'encode{2 * l + 1}', f'm{l}', 0, c1_dst, c1_coff, ch[l - 1], l, cout=ch[l], bm=bm))
        if v0:
            ops.append(_op(CONV, f'encode{2 * l + 2}', cat, p, e, 0, ch[l], l, cout=ch[l], bm=bm))
            ops.append(_op(POOL, None, e, 0, f'm{l + 1}', 0, p, l, bm=bm))
        elif l < 3 or not siam or siam_mode != 'concat':
            ops.append(_op(CONV, f'encode{2 * l + 2}', e, 0, cat, p, ch[l], l, cout=ch[l], bm=bm))
            ops.append(_op(POOL, None, cat, p, f'm{l + 1}', 0, p, l, bm=bm))
        else:       # concat join: pooled current -> joincat [0, 8 nf), pooled previous -> [8 nf, 16 nf)
            ops.append(_op(CONV, f'encode{2 * l + 2}', e, 0, cat, p, ch[l], l, cout=ch[l], bm=bm))
            ops.append(_op(POOL, None, cat, p, 'joincat', 0, p, l))
            ops.append(_op(POOL, None, cat, p, 'joincat', p, p, l, src_img0=1))
    mid_src = 'm4'
    if siam and siam_mode == 'concat':
        ops.append(_op(CONV, 'conv_concat', 'joincat', 0, 'join', 0, 2 * ch[3], 4,
                       segs=[(0, ch[3], 0), (ch[3], ch[3], pad16(ch[3]))], cout=ch[3]))
        mid_src = 'join'
    elif siam and siam_mode in ('max', 'corr'):
        ops.append(_op(MAXJOIN if siam_mode == 'max' else XCORR, None, 'm4', 0, 'join', 0, pad16(ch[3]), 4))
        mid_src = 'join'
    ops.append(_op(CONV, 'middle_conv1', mid_src, 0, 'mid1', 0, ch[3], 4, cout=ch[4]))
    ops.append(_op(CONV, 'middle_conv2', 'mid1', 0, 'mid2', 0, ch[4], 4, cout=ch[4]))
    prev, prev_c = 'mid2', ch[4]
    for l in range(3, -1, -1):
        k, cat, p = 3 - l, f'cat{4 - l}', pad16(ch[l])
        ops.append(_op(UP, f'up{k + 1}', prev, 0, cat, 0, prev_c, l + 1, cout=ch[l]))
        if att:
            ops.append(_op(GATE, f'attention{k + 1}', cat, 0, f'psi{4 - l}', 0, 2 * ch[l], l,
                           segs=[(0, ch[l], 0), (ch[l], ch[l], p)], cout=ch[l] // 2))
            ops.append(_op(MULPSI, None, f'psi{4 - l}', 0, cat, p, p, l))
            segs = [(0, ch[l], p), (ch[l], ch[l], 0)]        # cat((attention, up)): gated skip first
        else:
            segs = [(0, ch[l], 0), (ch[l], ch[l], p)]
        ops.append(_op(CONV, f'decode{2 * k + 1}', cat, 0, da[l], 0, 2 * ch[l], l, segs=segs, cout=ch[l]))
        if l > 0 or v0:
            ops.append(_op(CONV, f'decode{2 * k + 2}', da[l], 0, db[l], 0, ch[l], l, cout=ch[l]))
            prev, prev_c = db[l], ch[l]
        else:
            ops.append(_op(HEAD, 'decode8', da[0], 0, None, 0, ch[0], 0, cout=ch[0]))
    if v0:          # decode9: 3x3 block n_filter -> 1, then the 1 -> 1 head
        ops.append(_op(HEAD, 'decode9', db[0], 0, None, 0, ch[0], 0, cout=1))
    return bufs, ops, ('output_layers' if kind == 'mo2d' else 'final.0'), (0.0 if v0 else 0.1)


def _program_nested(kind, nf):
    """U-Net++ (MultiOutputNestedUNet / _3Levels): the last branch of net_build. Level l's nodes share ONE buffer
    x{l}: the up-sampling slot [0, upw[l]) first, node j at upw[l] + j * pc[l]; every node's first conv writes v{l}."""
    bufs, ops = {}, []
    lv = 4 if kind == 'nested2d' else 3
    ch = [nf << l for l in range(lv + 1)]
    pc = [pad16(c) for c in ch]
    upw = [pc[l + 1] if l < lv else 0 for l in range(lv + 1)]
    for l in range(lv + 1):
        j_max = lv - l
        bufs[f'x{l}'] = (l, upw[l] + (j_max if l == 0 else j_max + 1) * pc[l], 1)
        bufs[f'v{l}'] = (l, pc[l], 1)
        if l < lv:
            bufs[f'm{l + 1}'] = (l + 1, pc[l], 1)

    def keys(node, which):
        return (f'{node}.conv{which}', f'{node}.bn{which}')
    for s in range(lv + 1):
        node = f'conv{s}_0'
        if s == 0:
            ops.append(_op(FIRST, node + '.conv1', None, 0, 'v0', 0, 1, 0, cout=ch[0], keys=keys(node, 1)))
        else:
            ops.append(_op(CONV, node + '.conv1', f'm{s}', 0, f'v{s}', 0, ch[s - 1], s, cout=ch[s], keys=keys(node, 1)))
        ops.append(_op(CONV, node + '.conv2', f'v{s}', 0, f'x{s}', upw[s], ch[s], s, cout=ch[s], keys=keys(node, 2)))
        if s < lv:
            ops.append(_op(POOL, None, f'x{s}', upw[s], f'm{s + 1}', 0, pc[s], s))
        for j in range(1, s + 1):
            l = s - j
            node = f'conv{l}_{j}'
            ops.append(_op(UPBILINEAR, None, f'x{l + 1}', upw[l + 1] + (j - 1) * pc[l + 1], f'x{l}', 0, pc[l + 1],
                           l + 1))
            segs = [(k * ch[l], ch[l], upw[l] + k * pc[l]) for k in range(j)] + [(j * ch[l], ch[l + 1], 0)]
            ops.append(_op(CONV, node + '.conv1', f'x{l}', 0, f'v{l}', 0, j * ch[l] + ch[l + 1], l, segs=segs,
                           cout=ch[l], keys=keys(node, 1)))
            if l == 0 and j == lv:
                ops.append(_op(HEAD, node + '.conv2', 'v0', 0, None, 0, ch[0], 0, cout=ch[0], keys=keys(node, 2)))
            else:
                ops.append(_op(CONV, node + '.conv2', f'v{l}', 0, f'x{l}', upw[l] + j * pc[l], ch[l], l, cout=ch[l],
                               keys=keys(node, 2)))
    return bufs, ops, 'output_layers', 0.1


def program(kind, nf, interp=False, siam_mode='concat'):
    """(buffers {name: (level, channels, streams)}, ops, head param prefix, LeakyReLU slope) of net_build (in_channels
    1). segs: the layer's (logical start, count, physical start) input segments."""
    if kind in ('unet2d', 'attunet2d', 'siam2d', 'unet2d_v0', 'mo2d'):
        return _program_unet2d(kind, nf, siam_mode)
    if kind in ('nested2d', 'nested2d_3l'):
        return _program_nested(kind, nf)
    # UNet3D / MultiOutputUnet3D
    bufs, ops = {}, []
    tri = kind == 'unet3d' and interp
    h = nf // 2
    c_in, c_a = [1, nf, 2 * nf, 4 * nf], [h, nf, 2 * nf, 4 * nf]
    c_b, up_c = [nf, 2 * nf, 4 * nf, 8 * nf], [2 * nf, 4 * nf, 8 * nf]
    dec_out, dec_mid = [h, 2 * nf, 4 * nf], [nf, 2 * nf, 4 * nf]
    for l in range(3):
        bufs[f'e{2 * l + 1}'] = (l, pad16(c_a[l]), 1)
        bufs[f'cat{3 - l}'] = (l, pad16(up_c[l]) + pad16(c_b[l]), 1)
        bufs[f'm{l + 1}'] = (l + 1, pad16(c_b[l]), 1)
    bufs['mid1'], bufs['mid2'] = (3, pad16(c_a[3]), 1), (3, pad16(c_b[3]), 1)
    da, db, upt = {}, {}, {}
    for l in range(2, -1, -1):
        da[l] = f'd{2 * (2 - l) + 1}'
        bufs[da[l]] = (l, pad16(dec_mid[l]), 1)
        if l > 0:
            db[l] = f'd{2 * (2 - l) + 2}'
            bufs[db[l]] = (l, pad16(dec_out[l]), 1)
        if interp and not tri:
            upt[l] = f'upn{3 - l}'
            bufs[upt[l]] = (l, pad16(up_c[l]), 1)
    for l in range(3):
        e, cat, off = f'e{2 * l + 1}', f'cat{3 - l}', pad16(up_c[l])
        if l == 0:
            ops.append(_op(FIRST, 'encode1', None, 0, e, 0, 1, 0, cout=c_a[0]))
        else:
            ops.append(_op(CONV, f'encode{2 * l + 1}', f'm{l}', 0, e, 0, c_in[l], l, cout=c_a[l]))
        ops.append(_op(CONV, f'encode{2 * l + 2}', e, 0, cat, off, c_a[l], l, cout=c_b[l]))
        ops.append(_op(POOL, None, cat, off, f'm{l + 1}', 0, pad16(c_b[l]), l, pool_mode=1 if upt else 0))
    ops.append(_op(CONV, 'middle_conv1', 'm3', 0, 'mid1', 0, c_in[3], 3, cout=c_a[3]))
    ops.append(_op(CONV, 'middle_conv2', 'mid1', 0, 'mid2', 0, c_a[3], 3, cout=c_b[3]))
    prev, prev_c = 'mid2', c_b[3]
    for l in range(2, -1, -1):
        k, cat = 2 - l, f'cat{3 - l}'
        if tri:
            ops.append(_op(UPTRI, None, prev, 0, cat, 0, pad16(prev_c), l + 1))
        elif not interp:
            ops.append(_op(UP, f'up{k + 1}', prev, 0, cat, 0, prev_c, l + 1, cout=prev_c))
        else:
            ops.append(_op(UPNEAREST, None, prev, 0, upt[l], 0, pad16(prev_c), l + 1))
            ops.append(_op(CONV, f'up{k + 1}_conv', upt[l], 0, cat, 0, prev_c, l, cout=prev_c))
        ops.append(_op(CONV, f'decode{2 * k + 1}', cat, 0, da[l], 0, up_c[l] + c_b[l], l,
                       segs=[(0, up_c[l], 0), (up_c[l], c_b[l], pad16(up_c[l]))], cout=dec_mid[l]))
        if l > 0:
            ops.append(_op(CONV, f'decode{2 * k + 2}', da[l], 0, db[l], 0, dec_mid[l], l, cout=dec_out[l]))
            prev, prev_c = db[l], dec_out[l]
        else:
            ops.append(_op(HEAD, 'decode6', da[0], 0, None, 0, dec_mid[0], 0, cout=dec_out[0]))
    return bufs, ops, ('output_layers' if kind == 'mo3d' else 'final'), 0.1


def _phys(segs):
    idx = []
    for lstart, count, pstart in sorted(segs):
        idx.extend(range(pstart, pstart + count))
    return idx


def _src_channels(o):
    """Channel range [lo, hi) of the source buffer that op o reads."""
    if o['kind'] in (CONV, HEAD, GATE):
        return o['src_coff'], o['src_coff'] + max(p + n for _, n, p in o['segs'])
    return o['src_coff'], o['src_coff'] + o['c']


def _dst_channels(o):
    c = o['cout'] if o['kind'] in (CONV, UP, FIRST) else o['c']
    return o['dst_coff'], o['dst_coff'] + pad16(c)


# ------------------------------------------------------------------------------------------------ state dicts
def _model(kind, nf, interp, heads, siam_mode='concat'):
    from bio_image_unet_b200.multi_output_unet import (MultiOutputNestedUNet, MultiOutputNestedUNet_3Levels,
                                                       MultiOutputUnet)
    from bio_image_unet_b200.multi_output_unet3d import MultiOutputUnet3D
    from bio_image_unet_b200.siam_unet import Siam_UNet
    from bio_image_unet_b200.unet import AttentionUnet, Unet
    from bio_image_unet_b200.unet.unet_v0 import Unet_v0
    from bio_image_unet_b200.unet3d import UNet3D
    spec = {name: {'channels': c, 'activation': a} for name, c, a in heads}
    if kind == 'unet2d':
        return Unet(n_filter=nf)
    if kind == 'attunet2d':
        return AttentionUnet(n_filter=nf)
    if kind == 'siam2d':
        return Siam_UNet(n_filter=nf, mode=siam_mode)
    if kind == 'unet2d_v0':
        return Unet_v0(n_filter=nf)
    if kind == 'mo2d':
        return MultiOutputUnet(1, spec, nf)
    if kind == 'nested2d':
        return MultiOutputNestedUNet(1, spec, nf)
    if kind == 'nested2d_3l':
        return MultiOutputNestedUNet_3Levels(1, spec, nf)
    if kind == 'unet3d':
        return UNet3D(n_filter=nf, use_interpolation=interp) if interp else UNet3D(n_filter=nf)
    return MultiOutputUnet3D(1, spec, nf, interp)


def stress_state_dict(kind, nf, seed, interp=False, heads=(('', 1, 'sigmoid'),), siam_mode='concat'):
    """Kaiming weights and randomised BatchNorm statistics on the product's own module class."""
    torch.manual_seed(seed)
    sd = _model(kind, nf, interp, heads, siam_mode).state_dict()
    g = torch.Generator().manual_seed(seed)
    for k, v in sd.items():
        if k.endswith('num_batches_tracked'):
            continue
        if v.dim() > 1:
            fan_in = v.shape[0] if k.startswith('up') and 'conv' not in k else v[0].numel()
            sd[k] = torch.randn(v.shape, generator=g) * (2.0 / fan_in) ** 0.5
        elif k.endswith('running_var') or k.endswith('.1.weight') or k.endswith(('.bn1.weight', '.bn2.weight')):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
    return sd


# ------------------------------------------------------------------------------------------------ the check
class _Run:
    def __init__(self, eng, kind, nf, sd, inputs, in_float, val, u8, precision, imgs, heads, head_prefix, bufs, slope,
                 shared):
        self.eng, self.kind, self.nf, self.sd, self.precision = eng, kind, nf, sd, precision
        self.dims = 2 if kind in KINDS_2D else 3
        self.fmt = R.operand_format(precision)
        self.inputs, self.in_float, self.val, self.u8, self.imgs = inputs, in_float, val, u8, imgs
        self.heads, self.head_prefix, self.bufs, self.slope = heads, head_prefix, bufs, slope
        self.batch, self.shared = eng.batch, shared
        self.cache = {}
        self.saved = {}
        self.min_c = 0.0
        self.xcorr_c = 0.0

    def images(self, name):
        """Number of images a buffer holds: B, 2 B for a twin-encoder buffer, B + shared with the shared encoder."""
        bm = self.bufs[name][2]
        return self.batch + self.shared if (bm == 2 and self.shared > 0) else self.batch * bm

    def base(self, name, stream):
        """First image of a stream of a buffer (stream_img0 in net.cu)."""
        if self.bufs[name][2] == 2 and self.shared > 0:
            return self.shared if stream == 0 else 0
        return stream * self.batch

    def op_images(self, o, which):
        """Images of buffer o[which] ('src' / 'dst') the checked images of op o read / write."""
        name = o[which]
        if o['bm'] == 2 or (o['kind'] == FIRST and self.shared > 0 and o['src_img0'] == 0):
            # both streams (the shared encoder's first conv covers all unique tiles in its first op)
            return sorted({self.base(name, s) + i for s in (0, 1) for i in self.imgs})
        return [self.base(name, o[which + '_img0']) + i for i in self.imgs]

    def act(self, name):
        """Stored activation buffer (all its images), channels-last float32 on the GPU ((N, H, W, C) in 2D)."""
        if name not in self.cache:
            level, ctot, _ = self.bufs[name]
            a = torch.from_numpy(self.eng.debug_activation(name, ctot, level, images=self.images(name))).cuda()
            self.cache[name] = a[:, 0] if self.dims == 2 else a
        return self.cache[name]

    def psi(self, name):
        level, _, _ = self.bufs[name]
        d, h, w = self.eng.tile
        dd = max(d >> level, 1) if self.dims == 3 else 1
        host = np.empty(self.eng.batch * dd * (h >> level) * (w >> level), dtype=np.float32)
        from bio_image_unet_b200 import _lib
        torch.cuda.synchronize()
        _lib.check(self.eng.lib.biu_net_debug_copy(self.eng.handle, name.encode(), _lib.ptr(self.eng.workspace),
                                                   host.ctypes.data_as(ctypes.c_void_p), host.nbytes))
        return torch.from_numpy(host.reshape(self.eng.batch, h >> level, w >> level)[self.imgs]).cuda()

    def op_weights(self, o, tc):
        w, scale, shift = R.fold_bn(self.sd, *o['keys'])
        return (R.round_to(w, self.fmt) if tc else w), scale, shift

    def note_c(self, c):
        self.min_c = max(self.min_c, c)

    def conv_ref(self, o, fallback):
        """(S, A, scale, shift) of a Conv + BN op from the stored input."""
        tc = self.precision != 'fp32' and not fallback
        w, scale, shift = self.op_weights(o, tc)
        x = self.act(o['src'])[self.op_images(o, 'src')][..., [o['src_coff'] + p for p in _phys(o['segs'])]]
        s, a = R.conv_sums(x, w, self.dims)
        return s, a, scale, shift

    def out(self, o, c):
        return self.act(o['dst'])[self.op_images(o, 'dst')][..., o['dst_coff']:o['dst_coff'] + c]

    def src(self, o, c):
        return self.act(o['src'])[self.op_images(o, 'src')][..., o['src_coff']:o['src_coff'] + c]


def _check_op(run, i, o, fallback, rows_on):
    dims, fmt, slope, what = run.dims, run.fmt, run.slope, f"op {i} {o['layer'] or ''} ({o['kind']})"
    if o['kind'] == FIRST:
        dst_imgs = run.op_images(o, 'dst')
        x = run.inputs[dst_imgs].float().movedim(1, -1)       # (N, [D,] H, W, 1) raw uint8 values or float32 tiles
        # 2D, tensor-core mode, uint8 tiles, 16 / 32 channels, W >= 128: the row kernel's first mode
        # (conv_first_rows_supported); otherwise, and always in 3D or on float32 tiles, the CUDA-core first conv
        first_rows = run.precision != 'fp32' and dims == 2 and pad16(o['cout']) in (16, 32) and \
            x.shape[2] >= 128 and rows_on and not run.in_float
        w, scale, shift = R.fold_bn(run.sd, *o['keys'])
        if first_rows:       # raw uint8 times the rounded weights, scale_first = fp32(scale) / 255.0f in the epilogue
            w, scale = R.round_to(w, fmt), (scale / torch.tensor(255.0)).float()
        elif not run.in_float:   # float32(u8) / 255 times the fp32 weights; float32 tiles are used as they are
            x = (x.float() / torch.tensor(255.0, device=x.device)).float()
        s, a = R.conv_sums(x, w, dims)
        lo, hi = R.interval(s, a, scale, shift, slope, fmt, R.C_GPU)
        got = run.out(o, o['cout'])
        R.check_interval(got, lo, hi, what + (' first mode' if first_rows else ' CUDA-core'), index=dst_imgs)
        run.note_c(R.min_c(got, s, a, scale, shift, slope, fmt))
        return
    if o['kind'] == CONV:
        s, a, scale, shift = run.conv_ref(o, fallback)
        lo, hi = R.interval(s, a, scale, shift, slope, fmt, R.C_GPU)
        got = run.out(o, o['cout'])
        R.check_interval(got, lo, hi, what, index=run.op_images(o, 'dst'))
        run.note_c(R.min_c(got, s, a, scale, shift, slope, fmt))
        return
    if o['kind'] == HEAD:
        s, a, scale, shift = run.conv_ref(o, fallback)
        # contract of the value v the fused head reads: the tcgen05 epilogues feed the fp32 value (the row and halo
        # kernels tf32-round it in tf32 mode, the per-tap kernel does not); the CUDA-core fallback stores the
        # activation in the storage format first and the head kernel reads that
        vfmts = [fmt] if (fallback or run.precision == 'fp32') else (['fp32', 'tf32'] if fmt == 'tf32' else ['fp32'])
        bounds = [R.interval(s, a, scale, shift, slope, f, R.C_GPU) for f in vfmts]
        vlo = torch.stack([b[0] for b in bounds]).amin(0)
        vhi = torch.stack([b[1] for b in bounds]).amax(0)
        row = 0
        got = run.val[run.imgs].movedim(1, -1)
        for hname, hc, hact in run.heads:
            pre = run.head_prefix + ('.' + hname if run.head_prefix == 'output_layers' else '')
            hw = run.sd[pre + '.weight'].reshape(hc, -1).float()
            hb = run.sd[pre + '.bias'].float()
            lo, hi = R.head_interval(vlo, vhi, hw, hb, hact)
            g = got[..., row:row + hc]
            R.check_interval(g, lo.float(), hi.float(), f'{what} head {hname!r}', index=run.imgs, atol=1e-6)
            if hact == 'sigmoid':
                want = (g * torch.tensor(255.0, device=g.device)).to(torch.uint8)
                u8 = run.u8[run.imgs].movedim(1, -1)[..., row:row + hc].to(g.device)
                assert torch.equal(u8, want), f'{what}: out_u8 != uint8(out_val * 255)'
            row += hc
        return
    if o['kind'] == UP:
        tc = run.precision != 'fp32' and not fallback
        w = run.sd[o['layer'] + '.weight'].float()
        bias = run.sd[o['layer'] + '.bias'].float()
        x = run.src(o, o['c'])
        s, a = R.up_sums(x, R.round_to(w, fmt) if tc else w, dims)
        ones = torch.ones_like(bias)
        lo, hi = R.interval(s, a, ones, bias, 1.0, fmt, R.C_GPU)
        got = run.out(o, o['cout'])
        R.check_interval(got, lo, hi, what, index=run.op_images(o, 'dst'))
        run.note_c(R.min_c(got, s, a, ones, bias, 1.0, fmt))
        return
    if o['kind'] in (POOL, UPNEAREST):
        x = run.src(o, o['c'])
        if o['kind'] == UPNEAREST:
            ref = R.nearest_x2(x, dims)
        elif o['pool_mode'] == 1:
            ref = x[:, ::2, ::2, ::2] if dims == 3 else x[:, ::2, ::2]
        else:
            ref = R.maxpool(x, dims)
        got = run.out(o, o['c'])
        assert torch.equal(got, ref), f'{what}: {int((got != ref).sum())} values differ'
        return
    if o['kind'] == UPTRI:
        x = run.src(o, o['c'])
        s, a = R.trilinear_x2(x)
        z = torch.zeros(o['c'])
        lo, hi = R.interval(s, a, torch.ones(o['c']), z, 1.0, fmt, c=16.0)
        got = run.out(o, o['c'])
        R.check_interval(got, lo, hi, what, index=run.imgs)
        return
    if o['kind'] == UPBILINEAR:
        x = run.src(o, o['c'])
        s, a = R.bilinear_x2(x)
        z = torch.zeros(o['c'])
        lo, hi = R.interval(s, a, torch.ones(o['c']), z, 1.0, fmt, c=16.0)
        got = run.out(o, o['c'])
        R.check_interval(got, lo, hi, what, index=run.imgs)
        return
    if o['kind'] in (MAXJOIN, XCORR):
        emb = run.act(o['src'])[..., :o['c']]
        cur = emb[[run.base(o['src'], 0) + i for i in run.imgs]]
        prev = emb[[run.base(o['src'], 1) + i for i in run.imgs]]
        got = run.out(o, o['c'])
        if o['kind'] == MAXJOIN:
            ref = R.max_join(cur, prev)
            assert torch.equal(got, ref), f'{what}: {int((got != ref).sum())} values differ'
            return
        s, a, n = R.xcorr_sums(cur, prev)
        lo, hi = R.xcorr_interval(s, a, n, fmt)
        R.check_interval(got, lo, hi, what, ref=s, index=run.imgs)
        run.xcorr_c = max(run.xcorr_c, R.xcorr_min_c(got, s, a, n, fmt))
        return
    raise AssertionError(f'no reference for op kind {o["kind"]}')


def _check_gate(run, i, o, fallback):
    """Attention gate: psi = sigmoid(psi_w . ReLU(W [up | skip] + shift) + psi_b) from the stored concat buffer. The
    skip half is kept for the mul_psi that follows (it overwrites it in place)."""
    l = run.bufs[o['src']][0]
    c = run.nf << l
    p = pad16(c)
    xs = run.act(o['src'])[run.imgs]
    x = torch.cat([xs[..., :c], xs[..., p:p + c]], -1)
    w, gshift, gw, gb = R.fold_gate(run.sd, o['layer'], c)
    tc = run.precision != 'fp32' and not fallback
    wt = R.round_to(w, run.fmt) if tc else w
    sg, ag = R.gemm_sums(x, wt)
    vfmts = [run.fmt] if (fallback or run.precision == 'fp32') else (['fp32', 'tf32'] if run.fmt == 'tf32' else ['fp32'])
    ones = torch.ones_like(gshift)
    bounds = [R.interval(sg, ag, ones, gshift, 0.0, f, R.C_GPU) for f in vfmts]
    vlo = torch.stack([b[0] for b in bounds]).amin(0)
    vhi = torch.stack([b[1] for b in bounds]).amax(0)
    lo, hi = R.head_interval(vlo, vhi, gw[None], gb, 'sigmoid')
    psi = run.psi(o['dst'])
    R.check_interval(psi[..., None], lo.float(), hi.float(), f'op {i} {o["layer"]} psi', index=run.imgs, atol=1e-6)
    run.saved[i + 1] = (xs[..., p:p + c].clone(), psi.clone())


def _check_mulpsi(run, i, o):
    """skip * psi in fp32, one rounding to the storage format, in place: the skip as the gate's forward left it."""
    assert i in run.saved, f'op {i} mul_psi: its input was not captured at the gate'
    skip, psi0 = run.saved.pop(i)
    psi = run.psi(o['src'])
    assert torch.equal(psi, psi0), f'op {i} mul_psi: psi differs between two forwards of the same input'
    l = run.bufs[o['dst']][0]
    c = run.nf << l
    got = run.act(o['dst'])[run.imgs][..., o['dst_coff']:o['dst_coff'] + c]
    ref = R.round_to(skip * psi[..., None], run.fmt)
    R.check_interval(got, ref, ref, f'op {i} mul_psi', index=run.imgs)


def run_case(kind, nf, tile, batch, precision, imgs=None, interp=False, heads=(('', 1, 'sigmoid'),), ksplit=True,
             rows_on=True, seed=11, siam_mode='concat', siam_shared=0, float_input=False):
    """Plan, profiled forward, program check and every op against its reference.

    Ops whose input and output survive the forward are checked from that forward. Every other op k (its input or
    output is overwritten later: U-Net++'s shared v{l} buffers and up-sampling slots, the twin-encoder's second
    stream, e1 as a 3D K split's scratch, the CUDA-core head's staging buffer, the skip that mul_psi gates in place)
    is checked after a second forward of the same inputs that stops after op k (Engine.set_debug_stop). Nothing is
    skipped. ksplit: some 3D block splits K and uses e1 as its fp32 scratch."""
    from bio_image_unet_b200.engine import Engine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = stress_state_dict(kind, nf, seed, interp, heads, siam_mode)
    if kind == 'siam2d' and siam_mode == 'corr':
        # the correlation sums h * w products of two embeddings of size ~10: scale the last encoder block's BatchNorm
        # (and so the embedding, LeakyReLU being homogeneous) by 1 / sqrt(h * w) to keep fp16 below 65504
        k = ((tile[0] >> 4) * (tile[1] >> 4)) ** -0.5
        for key in ('encode8.1.weight', 'encode8.1.bias'):
            sd[key] = sd[key] * k
    g = torch.Generator().manual_seed(seed)
    twin = kind == 'siam2d' and siam_mode != 'control'
    shared = siam_shared if twin else 0
    n_in = batch + shared
    if float_input:
        tiles = torch.rand((n_in, 1, *tile), generator=g, dtype=torch.float32)
    else:
        tiles = torch.randint(0, 256, (n_in, 1, *tile), dtype=torch.uint8, generator=g)
    prev_tiles = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=g) if twin and not shared else None
    eng = Engine(kind, sd, nf, 1, list(heads), siam_mode=siam_mode, use_interpolation=interp, precision=precision,
                 device='cuda:0')
    try:
        eng.plan(batch, tile, siam_shared=shared)
        tiles_d = tiles.cuda()
        prev_d = prev_tiles.cuda() if prev_tiles is not None else None

        def forward():
            return eng.forward(tiles_d, prev_d, want_val=True, want_u8=True)
        eng.set_profile(1)
        val, u8 = forward()
        kinds, _ = eng.read_profile()
        eng.set_profile(0)
        bufs, ops, head_prefix, slope = program(kind, nf, interp, siam_mode)
        assert len(kinds) == len(ops), (len(kinds), len(ops))
        assert [k & 15 for k in kinds] == [o['kind'] for o in ops], kinds
        if imgs is None:
            imgs = sorted({0, batch // 2, batch - 1})
        # the tiles of every image of a first-conv buffer: [current | previous], or the unique tiles
        inputs = torch.cat([tiles, prev_tiles]) if prev_tiles is not None else tiles
        run = _Run(eng, kind, nf, sd, inputs.cuda(), float_input, val, u8, precision, imgs, heads, head_prefix, bufs,
                   slope, shared)
        # buffers whose content a later op replaced: (buffer, op index that writes it, channel range)
        clobber = [(o['dst'], j, *_dst_channels(o)) for j, o in enumerate(ops) if o['dst'] is not None]
        if run.dims == 3 and ksplit:
            j = next(j for j, o in enumerate(ops) if o['kind'] == CONV and o['level'] > 0)
            clobber.append(('e1', j, 0, 1 << 30))
        if kinds[-1] & 16:                   # the CUDA-core head stages the last activation in the first buffer
            clobber.append((list(bufs)[0], len(ops) - 1, 0, 1 << 30))

        def gone(buf, lo_c, hi_c, j):
            return any(b == buf and k > j and lo < hi_c and lo_c < hi for b, k, lo, hi in clobber)

        def survives(j, o):
            if o['kind'] in (GATE, MULPSI):          # mul_psi overwrites the gate's input in place
                return False
            if o['src'] is not None and gone(o['src'], *_src_channels(o), j):
                return False
            return o['dst'] is None or not gone(o['dst'], *_dst_channels(o), j)

        def check(j, o):
            fallback = bool(kinds[j] & 16)
            if o['kind'] == GATE:
                _check_gate(run, j, o, fallback)
            elif o['kind'] == MULPSI:
                _check_mulpsi(run, j, o)
            else:
                _check_op(run, j, o, fallback, rows_on)

        stopped = [j for j, o in enumerate(ops) if not survives(j, o)]
        checked = set()
        for j, o in enumerate(ops):
            if j not in stopped:
                check(j, o)
                checked.add(j)
        try:
            for j in stopped:
                eng.set_debug_stop(j)
                forward()
                run.cache.clear()
                check(j, ops[j])
                checked.add(j)
        finally:
            eng.set_debug_stop(-1)
        skipped = [f"op {j} {o['layer'] or ''} ({o['kind']})" for j, o in enumerate(ops) if j not in checked]
        return dict(kinds=kinds, skipped=skipped, stopped=len(stopped), min_c=run.min_c, xcorr_c=run.xcorr_c)
    finally:
        eng.close()


# ------------------------------------------------------------------------------------------------ cases
@pytest.fixture
def kernel_knob():
    """'default' | 'halo' (biu_set_rows_kernel(0)) | 'dual' (biu_set_rows_kernel(2)) | 'no_cta2' (biu_set_halo_cta2(0));
    the defaults are restored afterwards."""
    from bio_image_unet_b200 import _lib
    lib = _lib.load()

    def set_knob(name):
        lib.biu_set_rows_kernel({'halo': 0, 'dual': 2}.get(name, 1))
        lib.biu_set_halo_cta2(0 if name == 'no_cta2' else 1)
        return name != 'halo'
    yield set_knob
    lib.biu_set_rows_kernel(1)
    lib.biu_set_halo_cta2(1)


KNOBS = ['default', 'halo', 'dual', 'no_cta2']
PRECISIONS = ['bf16', 'fp16', 'tf32']
_MIN_C = {}


def _record(precision, res):
    """Print the largest accumulation allowance c any op needed so far in this precision (and, for the Siam
    cross-correlation, its c in units of gamma_n A), and require that every op of the program was checked."""
    _MIN_C[precision] = max(_MIN_C.get(precision, 0.0), res['min_c'])
    xc = f"; xcorr c = {res['xcorr_c']}" if res['xcorr_c'] else ''
    print(f"[layer-exact] {precision} max needed c = {_MIN_C[precision]}{xc}; stopped forwards: {res['stopped']}; "
          f"skipped: {res['skipped']}")
    assert res['skipped'] == [], res['skipped']


CASES_2D = {
    # first mode (W >= 128, 32 channels); row mode with a partial last strip (400 = 3 * 128 + 16); the wide N = 192
    # form at level 1 (64 channels, 200 px); halo kernel at level 2 (100 px, 128 channels); the per-tap small-plane
    # kernel with the batch packed into the box at level 4 (5 x 25, 512 channels)
    'unet2d_nf32_80x400': ('unet2d', 32, (80, 400), 1, None),
    # 16-channel row mode, ragged row blocks (48 rows), 16-px last strip (144 = 128 + 16), fused 2D pool
    'unet2d_nf16_48x144': ('unet2d', 16, (48, 144), 3, None),
    # halo CTA pairs at the wide levels; N split over 512 channels at level 4 (n_blk 256, non-resident weights)
    'unet2d_nf32_128x128': ('unet2d', 32, (128, 128), 6, None),
    # RB = 64 and both pipelines of the row kernel under the default rule (the flagship's shape); images 0 and 19
    'unet2d_nf32_512x512': ('unet2d', 32, (512, 512), 20, [0, 19]),
    # gate GEMM, psi head, mul_psi and the swapped concat order of the decode block
    'attunet_nf32_64x64': ('attunet2d', 32, (64, 64), 2, None),
    'attunet_nf16_128x144': ('attunet2d', 16, (128, 144), 1, None),
}


@pytest.mark.parametrize('knob', KNOBS)
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case', list(CASES_2D))
def test_2d_layers_exact(case, precision, knob, kernel_knob):
    kind, nf, tile, batch, imgs = CASES_2D[case]
    if case == 'unet2d_nf32_512x512' and knob != 'default':
        pytest.skip('the flagship shape runs under the default kernel choice only (its knobs are covered above)')
    rows_on = kernel_knob(knob)
    _record(precision, run_case(kind, nf, tile, batch, precision, imgs=imgs, rows_on=rows_on))


@pytest.mark.parametrize('case', ['unet2d_nf16_48x144', 'attunet_nf32_64x64'])
def test_2d_layers_exact_fp32(case):
    kind, nf, tile, batch, imgs = CASES_2D[case]
    res = run_case(kind, nf, tile, batch, 'fp32', imgs=imgs)
    assert all(k & 16 for k, o in zip(res['kinds'], program(kind, nf)[1]) if o['kind'] in (CONV, HEAD, UP))
    assert res['skipped'] == [], res['skipped']


CASES_3D = {
    # plane mode at level 0 with the fused MaxPool3d; K split of decode3 (96 -> 32)
    'unet3d_nf16_16x32x64': dict(kind='unet3d', nf=16, tile=(16, 32, 64), batch=2),
    # ragged 16 x 8 plane tiles; no K split, so encode1 / encode2 (e1) are checked
    'unet3d_nf32_16x48x40': dict(kind='unet3d', nf=32, tile=(16, 48, 40), batch=1, ksplit=False),
    # trilinear x2 up-sampling
    'unet3d_tri_nf16_16x32x64': dict(kind='unet3d', nf=16, tile=(16, 32, 64), batch=1, interp=True),
    # nearest up + up*_conv, fused multi-head with mixed activations
    'mo3d_nf16_16x32x96': dict(kind='mo3d', nf=16, tile=(16, 32, 96), batch=1, interp=True,
                               heads=(('a', 1, 'sigmoid'), ('b', 2, 'none'), ('c', 1, 'tanh'))),
}


@pytest.mark.parametrize('knob', KNOBS)
@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('case', list(CASES_3D))
def test_3d_layers_exact(case, precision, knob, kernel_knob):
    rows_on = kernel_knob(knob)
    _record(precision, run_case(precision=precision, rows_on=rows_on, **CASES_3D[case]))


@pytest.mark.parametrize('precision', PRECISIONS)
def test_unet3d_full_resolution_row_mode_child(precision):
    """Run only in the child process of test_unet3d_full_resolution_row_mode (BIU_ROWS_PLANE_FIRST=0)."""
    if os.environ.get('BIU_ROWS_PLANE_FIRST') != '0':
        pytest.skip('child of test_unet3d_full_resolution_row_mode')
    _record(precision, run_case('unet3d', 16, (8, 16, 128), 2, precision))


def test_unet3d_full_resolution_row_mode():
    """UNet3D nf 16, 8 x 16 x 128: with plane mode off the full-resolution blocks run in row mode, the epilogue pools
    every plane in (y, x) into pool_scratch and a second pass reduces the z pairs. The knob is read once per process,
    hence the child process."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, BIU_ROWS_PLANE_FIRST='0')
    r = subprocess.run([sys.executable, '-m', 'pytest', os.path.join(root, 'tests', 'test_gpu_layer_exact.py'), '-q',
                        '-m', 'gpu', '-k', 'test_unet3d_full_resolution_row_mode_child', '-p', 'no:cacheprovider'],
                       cwd=root, env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert '3 passed' in r.stdout, r.stdout[-500:]
