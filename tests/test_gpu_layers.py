"""Single layers of the CUDA kernels (through the C-ABI) against the exact single-op reference of tests/_layer_ref.py.

The operands are exactly representable on both sides, so every stored output must be the correctly rounded value of
the float64 result, up to the fp32 accumulation allowance (pools: bit-identical).
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from bio_image_unet_b200 import _lib
from tests import _layer_ref as R

pytestmark = pytest.mark.gpu


def _nhwc(x):  # (B,C,[D],H,W) -> channels-last contiguous
    if x.dim() == 4:
        return x.permute(0, 2, 3, 1).contiguous()
    return x.permute(0, 2, 3, 4, 1).contiguous()


def _nchw(x):
    if x.dim() == 4:
        return x.permute(0, 3, 1, 2).contiguous()
    return x.permute(0, 4, 1, 2, 3).contiguous()


def _sync_check():
    torch.cuda.synchronize()
    code = ctypes.c_uint(0)
    _lib.check(_lib.load().biu_device_fault(ctypes.byref(code)))
    assert code.value == 0, f'device fault {hex(code.value)}'


def _run_conv_tc(esz, B, cin, cout, D, H, W, k3d, seed, in_ctot=None, in_coff=0, out_ctot=None, out_coff=0):
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    lib = _lib.load()
    g = torch.Generator(device='cuda').manual_seed(seed)
    dt = torch.bfloat16 if esz == 2 else torch.float32
    in_ctot = in_ctot or cin
    out_ctot = out_ctot or cout
    dims3 = D > 1 or k3d
    shape = (B, in_ctot, D, H, W) if dims3 else (B, in_ctot, H, W)
    x = torch.randn(shape, device='cuda', generator=g).to(dt)
    kd = 3 if k3d else 1
    wshape = (cout, cin, kd, 3, 3) if dims3 else (cout, cin, 3, 3)
    w = (torch.randn(wshape, device='cuda', generator=g) / (cin * 9 * kd) ** 0.5).to(dt)
    if esz == 4:  # operands must be tf32-representable, as the engine guarantees
        x = (x.view(torch.int32) & ~0x1FFF).view(torch.float32)
        w = (w.view(torch.int32) & ~0x1FFF).view(torch.float32)
    scale = torch.rand(cout, device='cuda', generator=g) + 0.5
    shift = torch.randn(cout, device='cuda', generator=g) * 0.1
    x_cl = _nhwc(x)
    # packed weights [tap][cout][cin]
    if dims3:
        wp = w.permute(2, 3, 4, 0, 1).contiguous().view(kd * 9, cout, cin)
    else:
        wp = w.permute(2, 3, 0, 1).contiguous().view(9, cout, cin)
    out_shape = (B, D, H, W, out_ctot) if dims3 else (B, H, W, out_ctot)
    out = torch.zeros(out_shape, device='cuda', dtype=dt)
    rc = lib.biu_conv_tc(esz, _lib.ptr(x_cl), in_ctot, in_coff, cin, B, D, H, W, kd, 3, 3, _lib.ptr(wp), cout,
                         _lib.ptr(scale), _lib.ptr(shift), 0.1, _lib.ptr(out), out_ctot, out_coff, _lib.stream_ptr())
    _lib.check(rc, 'biu_conv_tc')
    _sync_check()
    s, a = R.conv_sums(x_cl[..., in_coff:in_coff + cin], w, 3 if dims3 else 2)
    lo, hi = R.interval(s, a, scale, shift, 0.1, 'bf16' if esz == 2 else 'tf32', R.C_GPU)
    return out[..., out_coff:out_coff + cout].float(), lo, hi


CASES_BF16 = [
    # B, cin, cout, D, H, W, k3d
    (2, 64, 64, 1, 32, 32, False),      # 128B swizzle
    (2, 32, 32, 1, 64, 64, False),      # 64B swizzle
    (3, 16, 16, 1, 16, 16, False),      # 32B swizzle
    (2, 128, 256, 1, 16, 16, False),    # N = 256
    (2, 256, 512, 1, 8, 8, False),      # N split over grid.y, box spans 2 images
    (1, 64, 32, 1, 24, 40, False),      # extents that are not powers of two (masked rows)
    (1, 32, 64, 1, 128, 128, False),    # box clipped to 32 wide
    (1, 32, 32, 8, 16, 16, True),       # 3D, 27 taps
    (1, 48, 16, 4, 8, 8, True),         # 3D, 3 chunks of 16
    (5, 512, 512, 1, 2, 2, False),      # tiny images, batch packed into the box
]


@pytest.mark.parametrize('case', CASES_BF16)
def test_conv_tc_bf16(case):
    B, cin, cout, D, H, W, k3d = case
    R.check_interval(*_run_conv_tc(2, B, cin, cout, D, H, W, k3d, seed=1), f'conv_tc bf16 {case}')


def test_conv_tc_bf16_concat_offsets():
    R.check_interval(*_run_conv_tc(2, 2, 64, 32, 1, 32, 32, False, seed=2, in_ctot=128, in_coff=64, out_ctot=96,
                                   out_coff=32), 'conv_tc bf16 concat offsets')


@pytest.mark.parametrize('case', [(2, 32, 32, 1, 32, 32, False), (1, 64, 128, 1, 16, 16, False),
                                  (1, 16, 16, 4, 8, 8, True), (2, 8, 16, 1, 16, 16, False)])
def test_conv_tc_tf32(case):
    B, cin, cout, D, H, W, k3d = case
    R.check_interval(*_run_conv_tc(4, B, cin, cout, D, H, W, k3d, seed=3), f'conv_tc tf32 {case}')


@pytest.mark.parametrize('dims,cin,cout', [(2, 64, 32), (2, 512, 256), (3, 32, 32), (2, 32, 16)])
def test_up_tc(dims, cin, cout):
    torch.backends.cudnn.allow_tf32 = False
    lib = _lib.load()
    g = torch.Generator(device='cuda').manual_seed(5)
    B, D, H, W = 2, (4 if dims == 3 else 1), 8, 16
    shape = (B, cin, D, H, W) if dims == 3 else (B, cin, H, W)
    x = torch.randn(shape, device='cuda', generator=g).bfloat16()
    wshape = (cin, cout, 2, 2, 2) if dims == 3 else (cin, cout, 2, 2)
    w = (torch.randn(wshape, device='cuda', generator=g) / cin ** 0.5).bfloat16()
    bias = torch.randn(cout, device='cuda', generator=g)
    nq = 8 if dims == 3 else 4
    # packed [q*cout + co][cin]
    wp = w.reshape(cin, cout, nq).permute(2, 1, 0).contiguous().view(nq * cout, cin)
    bias_rep = bias.repeat(nq).contiguous()
    oshape = (B, 2 * D, 2 * H, 2 * W, cout) if dims == 3 else (B, 2 * H, 2 * W, cout)
    out = torch.zeros(oshape, device='cuda', dtype=torch.bfloat16)
    x_cl = _nhwc(x)
    rc = lib.biu_up_tc(2, _lib.ptr(x_cl), cin, 0, cin, B, D, H, W, dims, _lib.ptr(wp), cout, _lib.ptr(bias_rep),
                       _lib.ptr(out), cout, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_up_tc')
    _sync_check()
    s, a = R.up_sums(_nhwc(x), w, dims)
    lo, hi = R.interval(s, a, torch.ones_like(bias), bias, 1.0, 'bf16', R.C_GPU)
    R.check_interval(out.float(), lo, hi, f'up_tc {dims}D {cin}->{cout}')


@pytest.mark.parametrize('esz', [2, 4])
def test_conv_direct(esz):
    torch.backends.cudnn.allow_tf32 = False
    lib = _lib.load()
    g = torch.Generator(device='cuda').manual_seed(7)
    dt = torch.bfloat16 if esz == 2 else torch.float32
    B, cin, cout, H, W = 2, 24, 40, 20, 28
    x = torch.randn(B, cin, H, W, device='cuda', generator=g).to(dt)
    w = torch.randn(cout, cin, 3, 3, device='cuda', generator=g) / (cin * 9) ** 0.5
    scale = torch.rand(cout, device='cuda', generator=g) + 0.5
    shift = torch.randn(cout, device='cuda', generator=g) * 0.1
    wp = w.permute(2, 3, 1, 0).contiguous().view(9, cin, cout)
    out = torch.zeros(B, H, W, cout, device='cuda', dtype=dt)
    x_cl = _nhwc(x)
    rc = lib.biu_conv_direct(esz, _lib.ptr(x_cl), cin, 0, cin, B, 1, H, W, 1, 3, 3, _lib.ptr(wp), cout,
                             _lib.ptr(scale), _lib.ptr(shift), 0.1, _lib.ptr(out), cout, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_conv_direct')
    _sync_check()
    # CUDA-core kernel: fp32 weights, fmaf accumulation; biu_conv_direct stores fp32 unrounded in the 4-byte format
    s, a = R.conv_sums(_nhwc(x), w, 2)
    lo, hi = R.interval(s, a, scale, shift, 0.1, 'bf16' if esz == 2 else 'fp32', R.C_GPU)
    R.check_interval(out.float(), lo, hi, f'conv_direct esz={esz}')


@pytest.mark.parametrize('dims,mode', [(2, 0), (3, 0), (3, 1)])
def test_pool2(dims, mode):
    lib = _lib.load()
    g = torch.Generator(device='cuda').manual_seed(9)
    B, C, D, H, W = 2, 32, (4 if dims == 3 else 1), 8, 12
    shape = (B, C, D, H, W) if dims == 3 else (B, C, H, W)
    x = torch.randn(shape, device='cuda', generator=g).bfloat16()
    oshape = (B, D // 2, H // 2, W // 2, C) if dims == 3 else (B, H // 2, W // 2, C)
    out = torch.zeros(oshape, device='cuda', dtype=torch.bfloat16)
    x_cl = _nhwc(x)
    rc = lib.biu_pool2(2, _lib.ptr(x_cl), C, 0, C, B, D, H, W, dims, mode, _lib.ptr(out), C, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_pool2')
    _sync_check()
    if mode == 0:
        ref = (F.max_pool3d if dims == 3 else F.max_pool2d)(x.float(), 2, 2)
    else:
        ref = F.interpolate(x.float(), scale_factor=0.5, mode='nearest')
    assert torch.equal(_nchw(out.float()), ref)
