"""Every op of the layer program against an exact single-op reference (tests/_layer_ref.py).

Each case plans a network, runs one profiled forward and recomputes every op whose input and output survive the
forward from the engine's OWN stored input, in float64: convolutions and transposed convolutions must give the
correctly rounded value (up to the fp32 accumulation allowance), pools and nearest up-sampling the exact maximum /
copy, trilinear up-sampling and the attention gate their interval, heads act(sum h_w v + h_b) within 1e-5. Nothing
compounds through the network, so a single wrong tap, rounding mode or scale index in any kernel variant fails here.

The program below mirrors net_build (bio_image_unet_b200/csrc/net.cu) for the families tested; the length and op
kinds of the engine's profile must match it, so a change of the program fails loudly.
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


# ------------------------------------------------------------------------------------------------ program mirror
def _op(kind, layer, src, src_coff, dst, dst_coff, c, level, segs=None, cout=None, pool_mode=0):
    return dict(kind=kind, layer=layer, src=src, src_coff=src_coff, dst=dst, dst_coff=dst_coff, c=c, level=level,
                segs=segs or [(0, c, 0)], cout=cout, pool_mode=pool_mode)


def program(kind, nf, interp=False):
    """(buffers {name: (level, channels)}, ops, head param prefix) of net_build for unet2d / attunet2d / unet3d / mo3d
    (in_channels 1). segs: the layer's (logical start, count, physical start) input segments."""
    bufs, ops = {}, []
    if kind in ('unet2d', 'attunet2d'):
        att = kind == 'attunet2d'
        ch = [nf << i for i in range(5)]
        for l in range(4):
            bufs[f'e{2 * l + 1}'] = (l, pad16(ch[l]))
            bufs[f'cat{4 - l}'] = (l, 2 * pad16(ch[l]))
            bufs[f'm{l + 1}'] = (l + 1, pad16(ch[l]))
        bufs['mid1'] = bufs['mid2'] = (4, pad16(ch[4]))
        da, db = {}, {}
        for l in range(3, -1, -1):
            da[l] = f'd{2 * (3 - l) + 1}'
            bufs[da[l]] = (l, pad16(ch[l]))
            if l > 0:
                db[l] = f'd{2 * (3 - l) + 2}'
                bufs[db[l]] = (l, pad16(ch[l]))
        for l in range(4):
            e, cat, p = f'e{2 * l + 1}', f'cat{4 - l}', pad16(ch[l])
            if l == 0:
                ops.append(_op(FIRST, 'encode1', None, 0, e, 0, 1, 0, cout=ch[0]))
            else:
                ops.append(_op(CONV, f'encode{2 * l + 1}', f'm{l}', 0, e, 0, ch[l - 1], l, cout=ch[l]))
            ops.append(_op(CONV, f'encode{2 * l + 2}', e, 0, cat, p, ch[l], l, cout=ch[l]))
            ops.append(_op(POOL, None, cat, p, f'm{l + 1}', 0, p, l))
        ops.append(_op(CONV, 'middle_conv1', 'm4', 0, 'mid1', 0, ch[3], 4, cout=ch[4]))
        ops.append(_op(CONV, 'middle_conv2', 'mid1', 0, 'mid2', 0, ch[4], 4, cout=ch[4]))
        prev, prev_c = 'mid2', ch[4]
        for l in range(3, -1, -1):
            k, cat, p = 3 - l, f'cat{4 - l}', pad16(ch[l])
            ops.append(_op(UP, f'up{k + 1}', prev, 0, cat, 0, prev_c, l + 1, cout=ch[l]))
            if att:
                bufs[f'psi{4 - l}'] = (l, None)
                ops.append(_op(GATE, f'attention{k + 1}', cat, 0, f'psi{4 - l}', 0, 2 * ch[l], l,
                               segs=[(0, ch[l], 0), (ch[l], ch[l], p)], cout=ch[l] // 2))
                ops.append(_op(MULPSI, None, f'psi{4 - l}', 0, cat, p, p, l))
                segs = [(0, ch[l], p), (ch[l], ch[l], 0)]        # cat((attention, up)): gated skip first
            else:
                segs = [(0, ch[l], 0), (ch[l], ch[l], p)]
            ops.append(_op(CONV, f'decode{2 * k + 1}', cat, 0, da[l], 0, 2 * ch[l], l, segs=segs, cout=ch[l]))
            if l > 0:
                ops.append(_op(CONV, f'decode{2 * k + 2}', da[l], 0, db[l], 0, ch[l], l, cout=ch[l]))
                prev, prev_c = db[l], ch[l]
            else:
                ops.append(_op(HEAD, 'decode8', da[0], 0, None, 0, ch[0], 0, cout=ch[0]))
        return bufs, ops, 'final.0'
    # UNet3D / MultiOutputUnet3D
    tri = kind == 'unet3d' and interp
    h = nf // 2
    c_in, c_a = [1, nf, 2 * nf, 4 * nf], [h, nf, 2 * nf, 4 * nf]
    c_b, up_c = [nf, 2 * nf, 4 * nf, 8 * nf], [2 * nf, 4 * nf, 8 * nf]
    dec_out, dec_mid = [h, 2 * nf, 4 * nf], [nf, 2 * nf, 4 * nf]
    for l in range(3):
        bufs[f'e{2 * l + 1}'] = (l, pad16(c_a[l]))
        bufs[f'cat{3 - l}'] = (l, pad16(up_c[l]) + pad16(c_b[l]))
        bufs[f'm{l + 1}'] = (l + 1, pad16(c_b[l]))
    bufs['mid1'], bufs['mid2'] = (3, pad16(c_a[3])), (3, pad16(c_b[3]))
    da, db, upt = {}, {}, {}
    for l in range(2, -1, -1):
        da[l] = f'd{2 * (2 - l) + 1}'
        bufs[da[l]] = (l, pad16(dec_mid[l]))
        if l > 0:
            db[l] = f'd{2 * (2 - l) + 2}'
            bufs[db[l]] = (l, pad16(dec_out[l]))
        if interp and not tri:
            upt[l] = f'upn{3 - l}'
            bufs[upt[l]] = (l, pad16(up_c[l]))
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
    return bufs, ops, ('output_layers' if kind == 'mo3d' else 'final')


def _phys(segs):
    idx = []
    for lstart, count, pstart in sorted(segs):
        idx.extend(range(pstart, pstart + count))
    return idx


# ------------------------------------------------------------------------------------------------ state dicts
def _model(kind, nf, interp, heads):
    from bio_image_unet_b200.multi_output_unet3d import MultiOutputUnet3D
    from bio_image_unet_b200.unet import AttentionUnet, Unet
    from bio_image_unet_b200.unet3d import UNet3D
    if kind == 'unet2d':
        return Unet(n_filter=nf)
    if kind == 'attunet2d':
        return AttentionUnet(n_filter=nf)
    if kind == 'unet3d':
        return UNet3D(n_filter=nf, use_interpolation=interp) if interp else UNet3D(n_filter=nf)
    spec = {name: {'channels': c, 'activation': a} for name, c, a in heads}
    return MultiOutputUnet3D(1, spec, nf, interp)


def stress_state_dict(kind, nf, seed, interp=False, heads=(('', 1, 'sigmoid'),)):
    """Kaiming weights and randomised BatchNorm statistics on the product's own module class."""
    torch.manual_seed(seed)
    sd = _model(kind, nf, interp, heads).state_dict()
    g = torch.Generator().manual_seed(seed)
    for k, v in sd.items():
        if k.endswith('num_batches_tracked'):
            continue
        if v.dim() > 1:
            fan_in = v.shape[0] if k.startswith('up') and 'conv' not in k else v[0].numel()
            sd[k] = torch.randn(v.shape, generator=g) * (2.0 / fan_in) ** 0.5
        elif k.endswith('running_var') or k.endswith('.1.weight'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
    return sd


# ------------------------------------------------------------------------------------------------ the check
class _Run:
    def __init__(self, eng, kind, nf, sd, tiles, val, u8, kinds, precision, imgs, heads, head_prefix, bufs):
        self.eng, self.kind, self.nf, self.sd, self.precision = eng, kind, nf, sd, precision
        self.dims = 3 if kind in ('unet3d', 'mo3d') else 2
        self.fmt = R.operand_format(precision)
        self.tiles, self.val, self.u8, self.kinds, self.imgs = tiles, val, u8, kinds, imgs
        self.heads, self.head_prefix, self.bufs = heads, head_prefix, bufs
        self.cache = {}
        self.min_c = 0.0

    def act(self, name):
        """Stored activation buffer, images self.imgs, channels-last float32 on the GPU ((N, H, W, C) in 2D)."""
        if name not in self.cache:
            level, ctot = self.bufs[name]
            a = torch.from_numpy(self.eng.debug_activation(name, ctot, level)[self.imgs]).cuda()
            self.cache[name] = a[:, 0] if self.dims == 2 else a
        return self.cache[name]

    def psi(self, name):
        level, _ = self.bufs[name]
        d, h, w = self.eng.tile
        dd = max(d >> level, 1) if self.dims == 3 else 1
        host = np.empty(self.eng.batch * dd * (h >> level) * (w >> level), dtype=np.float32)
        from bio_image_unet_b200 import _lib
        torch.cuda.synchronize()
        _lib.check(self.eng.lib.biu_net_debug_copy(self.eng.handle, name.encode(), _lib.ptr(self.eng.workspace),
                                                   host.ctypes.data_as(ctypes.c_void_p), host.nbytes))
        return torch.from_numpy(host.reshape(self.eng.batch, h >> level, w >> level)[self.imgs]).cuda()

    def op_weights(self, name, tc):
        w, scale, shift = R.fold_bn(self.sd, name + '.0', name + '.1')
        return (R.round_to(w, self.fmt) if tc else w), scale, shift

    def input_tiles(self):
        x = self.tiles[self.imgs].float()            # (N, 1, [D,] H, W) raw uint8 values
        return x.movedim(1, -1)

    def note_c(self, c):
        self.min_c = max(self.min_c, c)

    def conv_ref(self, o, fallback):
        """(S, A, scale, shift) of a Conv + BN op from the stored input."""
        tc = self.precision != 'fp32' and not fallback
        w, scale, shift = self.op_weights(o['layer'], tc)
        x = self.act(o['src'])[..., [o['src_coff'] + p for p in _phys(o['segs'])]]
        s, a = R.conv_sums(x, w, self.dims)
        return s, a, scale, shift


def _check_op(run, i, o, fallback, skip_in, skip_out, rows_on, skips):
    dims, fmt, what = run.dims, run.fmt, f"op {i} {o['layer'] or ''} ({o['kind']})"
    if o['kind'] == FIRST:
        if skip_out:
            skips.append(what)
            return
        x = run.input_tiles()
        # 2D, tensor-core mode, 16 / 32 channels, W >= 128: the row kernel's first mode (conv_first_rows_supported);
        # otherwise, and always in 3D, the CUDA-core first conv
        first_rows = run.precision != 'fp32' and dims == 2 and pad16(o['cout']) in (16, 32) and \
            x.shape[2] >= 128 and rows_on
        w, scale, shift = R.fold_bn(run.sd, 'encode1.0', 'encode1.1')
        if first_rows:       # raw uint8 times the rounded weights, scale_first = fp32(scale) / 255.0f in the epilogue
            w, scale = R.round_to(w, fmt), (scale / torch.tensor(255.0)).float()
        else:                # float32(u8) / 255 times the fp32 weights
            x = (x.float() / torch.tensor(255.0, device=x.device)).float()
        s, a = R.conv_sums(x, w, dims)
        lo, hi = R.interval(s, a, scale, shift, 0.1, fmt, R.C_GPU)
        got = run.act(o['dst'])[..., o['dst_coff']:o['dst_coff'] + o['cout']]
        R.check_interval(got, lo, hi, what + (' first mode' if first_rows else ' CUDA-core'), index=run.imgs)
        run.note_c(R.min_c(got, s, a, scale, shift, 0.1, fmt))
        return
    if o['kind'] == CONV:
        if skip_in or skip_out:
            skips.append(what)
            return
        s, a, scale, shift = run.conv_ref(o, fallback)
        lo, hi = R.interval(s, a, scale, shift, 0.1, fmt, R.C_GPU)
        got = run.act(o['dst'])[..., o['dst_coff']:o['dst_coff'] + o['cout']]
        R.check_interval(got, lo, hi, what, index=run.imgs)
        run.note_c(R.min_c(got, s, a, scale, shift, 0.1, fmt))
        return
    if o['kind'] == HEAD:
        if skip_in:
            skips.append(what)
            return
        s, a, scale, shift = run.conv_ref(o, fallback)
        # contract of the value v the fused head reads: the tcgen05 epilogues feed the fp32 value (the row and halo
        # kernels tf32-round it in tf32 mode, the per-tap kernel does not); the CUDA-core fallback stores the
        # activation in the storage format first and the head kernel reads that
        vfmts = [fmt] if (fallback or run.precision == 'fp32') else (['fp32', 'tf32'] if fmt == 'tf32' else ['fp32'])
        bounds = [R.interval(s, a, scale, shift, 0.1, f, R.C_GPU) for f in vfmts]
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
        if skip_out:
            skips.append(what)
            return
        tc = run.precision != 'fp32' and not fallback
        w = run.sd[o['layer'] + '.weight'].float()
        bias = run.sd[o['layer'] + '.bias'].float()
        x = run.act(o['src'])[..., o['src_coff']:o['src_coff'] + o['c']]
        s, a = R.up_sums(x, R.round_to(w, fmt) if tc else w, dims)
        ones = torch.ones_like(bias)
        lo, hi = R.interval(s, a, ones, bias, 1.0, fmt, R.C_GPU)
        got = run.act(o['dst'])[..., o['dst_coff']:o['dst_coff'] + o['cout']]
        R.check_interval(got, lo, hi, what, index=run.imgs)
        run.note_c(R.min_c(got, s, a, ones, bias, 1.0, fmt))
        return
    if o['kind'] in (POOL, UPNEAREST):
        if skip_in or skip_out:
            skips.append(what)
            return
        x = run.act(o['src'])[..., o['src_coff']:o['src_coff'] + o['c']]
        if o['kind'] == UPNEAREST:
            ref = R.nearest_x2(x, dims)
        elif o['pool_mode'] == 1:
            ref = x[:, ::2, ::2, ::2] if dims == 3 else x[:, ::2, ::2]
        else:
            ref = R.maxpool(x, dims)
        got = run.act(o['dst'])[..., o['dst_coff']:o['dst_coff'] + o['c']]
        assert torch.equal(got, ref), f'{what}: {int((got != ref).sum())} values differ'
        return
    if o['kind'] == UPTRI:
        x = run.act(o['src'])[..., o['src_coff']:o['src_coff'] + o['c']]
        s, a = R.trilinear_x2(x)
        z = torch.zeros(o['c'])
        lo, hi = R.interval(s, a, torch.ones(o['c']), z, 1.0, fmt, c=16.0)
        got = run.act(o['dst'])[..., o['dst_coff']:o['dst_coff'] + o['c']]
        R.check_interval(got, lo, hi, what, index=run.imgs)
        return
    raise AssertionError(f'no reference for op kind {o["kind"]}')


def _check_attention(run, ops, i, fallback, kinds):
    """Gate (op i), then mul_psi (op i + 1). The pre-gate skip half of the concat buffer is overwritten by mul_psi, so
    it is recomputed from its encoder block as the interval of values the engine may have stored there (one-ulp
    flips allowed), and carried through the gate GEMM as a box."""
    o = ops[i]
    l = run.bufs[o['src']][0]
    c = run.nf << l
    p = pad16(c)
    enc = next(e for e in ops if e['kind'] == CONV and e['dst'] == o['src'] and e['dst_coff'] == p)
    enc_fallback = bool(kinds[ops.index(enc)] & 16)
    s, a, scale, shift = run.conv_ref(enc, enc_fallback)
    slo, shi = R.interval(s, a, scale, shift, 0.1, run.fmt, R.C_GPU)
    up = run.act(o['src'])[..., :c].double()
    w, gshift, gw, gb = R.fold_gate(run.sd, o['layer'], c)
    tc = run.precision != 'fp32' and not fallback
    wt = R.round_to(w, run.fmt) if tc else w
    xmid = torch.cat([up, (slo.double() + shi.double()) / 2], -1)
    rad = torch.cat([torch.zeros_like(up), (shi.double() - slo.double()) / 2], -1)
    sg, ag = R.gemm_sums(xmid, wt)
    box = rad @ wt.double().abs().t().to(rad.device)
    vfmts = [run.fmt] if (fallback or run.precision == 'fp32') else (['fp32', 'tf32'] if run.fmt == 'tf32' else ['fp32'])
    ones = torch.ones_like(gshift)
    bl = [R.interval(sg - box, ag, ones, gshift, 0.0, f, R.C_GPU) for f in vfmts]
    bh = [R.interval(sg + box, ag, ones, gshift, 0.0, f, R.C_GPU) for f in vfmts]
    vlo = torch.stack([b[0] for b in bl]).amin(0)
    vhi = torch.stack([b[1] for b in bh]).amax(0)
    lo, hi = R.head_interval(vlo, vhi, gw[None], gb, 'sigmoid')
    psi = run.psi(o['dst'])
    R.check_interval(psi[..., None], lo.float(), hi.float(), f'op {i} {o["layer"]} psi', index=run.imgs, atol=1e-6)
    # mul_psi: skip * psi in fp32, one rounding to the storage format (psi >= 0 keeps the order)
    got = run.act(o['src'])[..., p:p + c]
    ps = psi[..., None]
    lo = R.round_to(slo * ps, run.fmt)
    hi = R.round_to(shi * ps, run.fmt)
    R.check_interval(got, lo, hi, f'op {i + 1} mul_psi', index=run.imgs)


def run_case(kind, nf, tile, batch, precision, imgs=None, interp=False, heads=(('', 1, 'sigmoid'),), ksplit=True,
             rows_on=True, seed=11):
    """Plan, profiled forward, program check and every op against its reference. ksplit: some 3D block splits K and
    uses e1 as its fp32 scratch (e1 and the ops reading / writing it are then not checked)."""
    from bio_image_unet_b200.engine import Engine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    sd = stress_state_dict(kind, nf, seed, interp, heads)
    g = torch.Generator().manual_seed(seed)
    tiles = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=g)
    eng = Engine(kind, sd, nf, 1, list(heads), use_interpolation=interp, precision=precision, device='cuda:0')
    try:
        eng.plan(batch, tile)
        eng.set_profile(1)
        val, u8 = eng.forward(tiles.cuda(), want_val=True, want_u8=True)
        kinds, _ = eng.read_profile()
        eng.set_profile(0)
        bufs, ops, head_prefix = program(kind, nf, interp)
        assert len(kinds) == len(ops), (len(kinds), len(ops))
        assert [k & 15 for k in kinds] == [o['kind'] for o in ops], kinds
        if imgs is None:
            imgs = sorted({0, batch // 2, batch - 1})
        run = _Run(eng, kind, nf, sd, tiles.cuda(), val, u8, kinds, precision, imgs, heads, head_prefix, bufs)
        dims = run.dims
        # buffers whose content a later op replaced: (buffer, op index after which it is gone, channel range)
        clobber = []
        for j, o in enumerate(ops):
            if o['dst'] is not None:
                c = o['cout'] if o['kind'] in (CONV, UP, FIRST) else o['c']
                clobber.append((o['dst'], j, o['dst_coff'], o['dst_coff'] + pad16(c)))
        if dims == 3 and ksplit:
            j = next(j for j, o in enumerate(ops) if o['kind'] == CONV and o['level'] > 0)
            clobber.append(('e1', j, 0, 1 << 30))
        if kinds[-1] & 16:                   # the CUDA-core head stages the last activation in the first buffer
            clobber.append((list(bufs)[0], len(ops) - 1, 0, 1 << 30))

        def gone(buf, coff, c, j):
            return any(b == buf and k > j and lo < coff + c and coff < hi for b, k, lo, hi in clobber)

        skips = []
        for j, o in enumerate(ops):
            fallback = bool(kinds[j] & 16)
            if o['kind'] == GATE:
                enc_src = run.bufs[o['src']][0]
                if gone(f'e{2 * enc_src + 1}', 0, 16, j):       # the skip cannot be recomputed
                    skips.append(f'op {j} {o["layer"]} + mul_psi')
                else:
                    _check_attention(run, ops, j, fallback, kinds)
                continue
            if o['kind'] == MULPSI:
                continue
            c_in = o['c'] if o['kind'] != CONV else max(p for _, n, p in o['segs']) + 16
            skip_in = o['src'] is not None and gone(o['src'], o['src_coff'], c_in, j)
            skip_out = o['dst'] is not None and gone(o['dst'], o['dst_coff'], pad16(o['cout'] or o['c']), j)
            _check_op(run, j, o, fallback, skip_in, skip_out, rows_on, skips)
        return dict(kinds=kinds, skipped=skips, min_c=run.min_c)
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
    _MIN_C[precision] = max(_MIN_C.get(precision, 0.0), res['min_c'])
    print(f"[layer-exact] {precision} max needed c = {_MIN_C[precision]}; skipped: {res['skipped']}")


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
