"""The fp16 precision mode on the GPU: fp16 tcgen05 operands (kind::f16, F16 A/B formats), fp32 accumulation and
epilogue, fp16 activation storage.

* golden parity of every model family in fp16 against the fixtures of the unmodified reference, within 1.5x what the
  reference's own fp16 arithmetic (torch.autocast(float16) / fp16-rounded operands, tests/_parity_fp16.py) moves the result,
  through the same test bodies the other precisions use;
* the tf32 gate (1e-3) on PyTorch's default init, and fp16 at most half bf16's mean error on a stress net;
* the BASELINE-size shapes with every layer on the tensor-core kernels (row kernel with first mode, wide blocks and
  fused pools, plane mode, K split, CTA pairs);
* the bit-identities the bf16 mode guarantees (CTA pairs, shared Siam encoder, pipelined 3D groups, fused pools);
* the single layers through the layer C-ABI with the fp16 element code (BIU_ESZ_FP16).
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from bio_image_unet_b200 import _lib
from oracle import models as omodels
from tests import _golden, _layer_ref, _parity_fp16
from tests import test_gpu_baseline_sizes as sizes
from tests import test_gpu_families as families
from tests import test_gpu_unet as unet

pytestmark = pytest.mark.gpu


@pytest.fixture(autouse=True)
def fp16_parity():
    """The test bodies shared with the other precisions ask tests/_parity.py for their bounds: answer 'fp16' there with
    the reference's fp16 arithmetic."""
    with _parity_fp16.extend_parity():
        yield

ESZ_FP16 = 3          # BIU_ESZ_FP16 (include/biu_b200.h)


# ---------------------------------------------------------------------------------------------------------------------
# golden fixtures of the reference, every family
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['unet_single', 'unet_all_invert', 'unet_first_u8', 'unet_small_reflect'])
def test_unet_golden_fp16(name, tmp_path):
    unet.test_predict_matches_reference_golden(name, 'fp16', tmp_path)


@pytest.mark.parametrize('name', ['attunet_single', 'unetv0_all'])
def test_attention_unet_and_unet_v0_golden_fp16(name, tmp_path):
    unet.test_variant_predict_matches_reference_golden(name, 'fp16', False, tmp_path)


@pytest.mark.parametrize('name', ['siam_concat', 'siam_max', 'siam_control_small', 'siam_corr'])
def test_siam_golden_fp16(name, tmp_path):
    families.test_siam_predict_matches_reference_golden(name, 'fp16', tmp_path)


@pytest.mark.parametrize('name', ['unet3d_overlap', 'unet3d_disjoint', 'unet3d_trilinear'])
def test_unet3d_golden_fp16(name, tmp_path):
    families.test_unet3d_predict_matches_reference_golden(name, 'fp16', tmp_path)


@pytest.mark.parametrize('name', ['mo3d_interp', 'mo3d_convt'])
def test_mo3d_golden_fp16(name, tmp_path):
    families.test_mo3d_predict_matches_reference_golden(name, 'fp16', tmp_path)


@pytest.mark.parametrize('name', ['mo2d_single_overlap', 'mo2d_all_pad', 'mo2d_first_holes'])
def test_mo2d_golden_fp16(name, tmp_path):
    families.test_mo2d_predict_matches_reference_golden(name, 'fp16', tmp_path)


@pytest.mark.parametrize('name', ['nested_single_overlap', 'nested3l_ds_all'])
def test_nested_golden_fp16(name, tmp_path):
    families.test_nested_predict_matches_reference_golden(name, 'fp16', tmp_path)


# ---------------------------------------------------------------------------------------------------------------------
# accuracy against the oracle
# ---------------------------------------------------------------------------------------------------------------------
def test_default_init_unet_within_tf32_gate():
    unet.test_engine_forward_matches_oracle('fp16', 'default', 32, (64, 64), 2)


def test_default_init_unet3d_within_tf32_gate():
    from bio_image_unet_b200.engine import Engine
    from bio_image_unet_b200.unet3d import UNet3D
    torch.manual_seed(16)
    sd = UNet3D(n_filter=16).state_dict()
    x_u8 = torch.randint(0, 256, (2, 1, 16, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(6))
    with torch.no_grad():
        ref = omodels.unet3d_forward(sd, x_u8.float() / 255)[0]
    eng = Engine('unet3d', sd, 16, 1, [('', 1, 'sigmoid')], precision='fp16', device='cuda:0')
    eng.plan(2, (16, 64, 64))
    val, _ = eng.forward(x_u8.cuda(), want_val=True)
    err = (val.cpu() - ref).abs().max().item()
    assert err <= _parity_fp16.NORTH_STAR, err
    assert eng.fallback_ops == 0
    eng.close()


def test_fp16_error_at_most_half_of_bf16():
    """Same stress Unet(32), same tiles: fp16 keeps 10 mantissa bits against bf16's 7."""
    from bio_image_unet_b200.engine import Engine
    tiles = torch.randint(0, 256, (2, 1, 128, 128), dtype=torch.uint8, generator=torch.Generator().manual_seed(8))
    sd = unet.unit_logit_state_dict(32, 132, tiles)
    with torch.no_grad():
        ref = omodels.unet_forward(sd, tiles.float() / 255)[0]
    err = {}
    for precision in ('bf16', 'fp16'):
        eng = Engine('unet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
        eng.plan(2, (128, 128))
        val, _ = eng.forward(tiles.cuda(), want_val=True)
        err[precision] = (val.cpu() - ref).abs().mean().item()
        assert eng.fallback_ops == 0
        eng.close()
    assert err['fp16'] <= 0.5 * err['bf16'], err


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE-size shapes: every layer on the tcgen05 kernels (fallback_ops == 0 is asserted inside)
# ---------------------------------------------------------------------------------------------------------------------
def test_cfg2_tiles_in_a_full_batch_fp16():
    sizes.test_cfg2_tiles_in_a_full_batch_match_oracle('fp16')


def test_cfg4_unet3d_patch_fp16():
    sizes.test_cfg4_unet3d_patch_matches_oracle('fp16')


# ---------------------------------------------------------------------------------------------------------------------
# bit-identities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def cta2_toggle():
    lib = _lib.load()
    yield lambda on: lib.biu_set_halo_cta2(int(on))
    lib.biu_set_halo_cta2(1)


@pytest.mark.parametrize('kind,n_filter,tile,batch', [('unet2d', 32, (128, 128), 6), ('unet2d', 16, (256, 64), 3),
                                                      ('unet3d', 32, (16, 32, 32), 2)])
def test_cta_pairs_match_single_cta_fp16(kind, n_filter, tile, batch, cta2_toggle):
    unet.test_cta_pairs_match_single_cta('fp16', kind, n_filter, tile, batch, cta2_toggle)


@pytest.mark.parametrize('mode', ['concat', 'max', 'corr'])
def test_siam_shared_encoder_is_bit_identical_fp16(mode):
    families.test_siam_shared_encoder_is_bit_identical(mode, 'fp16')


@pytest.mark.parametrize('tile', [(64, 64), (48, 80), (128, 32)])
def test_fused_maxpool_is_bit_identical_fp16(tile):
    unet.test_fused_maxpool_is_bit_identical('fp16', tile)


@pytest.mark.parametrize('add_patch', [0, 1])
def test_unet3d_pipelined_groups_equal_whole_volume_fp16(add_patch):
    from bio_image_unet_b200.unet3d import Session
    g = _golden.load('unet3d_overlap')
    sd, rd = _golden.state_dict(g), tuple(int(v) for v in g['resize_dim'])
    base = g['vol']
    reps = (-(-(5 * rd[0] + 3) // base.shape[0]), 1, 1)
    vol = np.tile(base, reps)[:5 * rd[0] + 3].copy()
    vol[::2] = vol[::2, ::-1]
    ses = Session({'state_dict': sd, 'n_filter': int(g['n_filter']), 'in_channels': 1, 'out_channels': 1}, rd,
                  add_patch=add_patch, clip_threshold=tuple(g['clip']), device='cuda:0', precision='fp16')
    piped = np.array(ses.predict(vol.copy()))
    assert ses.N_z >= 2
    plain = np.array(ses.predict(vol.copy(), keep=True))
    assert piped.std() > 0 and np.array_equal(piped, plain)
    ses.close()


# ---------------------------------------------------------------------------------------------------------------------
# single layers through the layer C-ABI (element code BIU_ESZ_FP16), against torch on the same fp16 operands
# ---------------------------------------------------------------------------------------------------------------------
def _nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous() if x.dim() == 4 else x.permute(0, 2, 3, 4, 1).contiguous()


def _nchw(x):
    return x.permute(0, 3, 1, 2).contiguous() if x.dim() == 4 else x.permute(0, 4, 1, 2, 3).contiguous()


def _sync_check():
    torch.cuda.synchronize()
    code = ctypes.c_uint(0)
    _lib.check(_lib.load().biu_device_fault(ctypes.byref(code)))
    assert code.value == 0, f'device fault {hex(code.value)}'


def _conv_tc_fp16(case, shift_gain=0.1, scale_gain=1.0):
    torch.backends.cudnn.allow_tf32 = False
    B, cin, cout, D, H, W, three = case
    g = torch.Generator(device='cuda').manual_seed(11)
    kd = 3 if three else 1
    x = torch.randn((B, cin, D, H, W) if three else (B, cin, H, W), device='cuda', generator=g).half()
    w = (torch.randn((cout, cin, kd, 3, 3) if three else (cout, cin, 3, 3), device='cuda', generator=g)
         / (cin * 9 * kd) ** 0.5).half()
    scale = (torch.rand(cout, device='cuda', generator=g) + 0.5) * scale_gain
    shift = torch.randn(cout, device='cuda', generator=g) * shift_gain
    wp = (w.permute(2, 3, 4, 0, 1) if three else w.permute(2, 3, 0, 1)).contiguous().view(kd * 9, cout, cin)
    out = torch.zeros((B, D, H, W, cout) if three else (B, H, W, cout), device='cuda', dtype=torch.float16)
    x_cl = _nhwc(x)
    rc = _lib.load().biu_conv_tc(ESZ_FP16, _lib.ptr(x_cl), cin, 0, cin, B, D, H, W, kd, 3, 3, _lib.ptr(wp), cout,
                                 _lib.ptr(scale), _lib.ptr(shift), 0.1, _lib.ptr(out), cout, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_conv_tc')
    _sync_check()
    # fp32 accumulation of the same operands, one fp16 rounding (nearest even, beyond +-65504 +-inf) of the stored value
    s, a = _layer_ref.conv_sums(_nhwc(x), w, 3 if three else 2)
    lo, hi = _layer_ref.interval(s, a, scale, shift, 0.1, 'fp16', _layer_ref.C_GPU)
    return out.float(), lo, hi


@pytest.mark.parametrize('case', [
    # B, cin, cout, D, H, W, 3D
    (2, 64, 64, 1, 32, 32, False),      # halo kernel, 128B swizzle, CTA pairs
    (3, 16, 16, 1, 16, 16, False),      # 32B swizzle
    (2, 128, 256, 1, 16, 16, False),    # N = 256
    (1, 64, 32, 1, 24, 40, False),      # extents that are not powers of two
    (5, 512, 512, 1, 2, 2, False),      # tiny planes: per-tap kernel, batch packed into the box
    (1, 32, 32, 8, 16, 16, True),       # 3D, 27 taps
])
def test_conv_tc_fp16(case):
    _layer_ref.check_interval(*_conv_tc_fp16(case), f'conv_tc fp16 {case}')


@pytest.mark.parametrize('case', [(2, 64, 64, 1, 32, 32, False),     # halo kernel
                                  (5, 512, 512, 1, 2, 2, False)])     # per-tap small-plane kernel
def test_conv_tc_fp16_overflow_is_inf(case):
    """DESIGN §5: fp16 stores do not saturate. A shift of about +-65000 and a scale of 2000 push part of the outputs
    past +-65504: they must be +-inf exactly where the correctly rounded value is, and correctly rounded elsewhere."""
    got, lo, hi = _conv_tc_fp16(case, shift_gain=40000.0, scale_gain=2000.0)
    _layer_ref.check_interval(got, lo, hi, f'conv_tc fp16 overflow {case}')
    assert bool(torch.isinf(got).any()) and bool(torch.isfinite(got).any()), 'the case must reach both sides of 65504'


@pytest.mark.parametrize('dims,cin,cout', [(2, 64, 32), (2, 512, 256), (3, 32, 32)])
def test_up_tc_fp16(dims, cin, cout):
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device='cuda').manual_seed(13)
    B, D, H, W = 2, (4 if dims == 3 else 1), 8, 16
    x = torch.randn((B, cin, D, H, W) if dims == 3 else (B, cin, H, W), device='cuda', generator=g).half()
    w = (torch.randn((cin, cout, 2, 2, 2) if dims == 3 else (cin, cout, 2, 2), device='cuda', generator=g)
         / cin ** 0.5).half()
    bias = torch.randn(cout, device='cuda', generator=g)
    nq = 8 if dims == 3 else 4
    wp = w.reshape(cin, cout, nq).permute(2, 1, 0).contiguous().view(nq * cout, cin)
    out = torch.zeros((B, 2 * D, 2 * H, 2 * W, cout) if dims == 3 else (B, 2 * H, 2 * W, cout), device='cuda',
                      dtype=torch.float16)
    # named, so that they outlive the launch: the caching allocator hands a freed temporary's memory to the next
    # allocation, and a copy queued before the kernel would overwrite its input
    x_cl = _nhwc(x)
    bias_rep = bias.repeat(nq).contiguous()
    rc = _lib.load().biu_up_tc(ESZ_FP16, _lib.ptr(x_cl), cin, 0, cin, B, D, H, W, dims, _lib.ptr(wp), cout,
                               _lib.ptr(bias_rep), _lib.ptr(out), cout, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_up_tc')
    _sync_check()
    s, a = _layer_ref.up_sums(_nhwc(x), w, dims)
    lo, hi = _layer_ref.interval(s, a, torch.ones_like(bias), bias, 1.0, 'fp16', _layer_ref.C_GPU)
    _layer_ref.check_interval(out.float(), lo, hi, f'up_tc fp16 {dims}D {cin}->{cout}')


def test_conv_direct_fp16():
    torch.backends.cudnn.allow_tf32 = False
    g = torch.Generator(device='cuda').manual_seed(17)
    B, cin, cout, H, W = 2, 24, 40, 20, 28
    x = torch.randn(B, cin, H, W, device='cuda', generator=g).half()
    w = torch.randn(cout, cin, 3, 3, device='cuda', generator=g) / (cin * 9) ** 0.5
    scale = torch.rand(cout, device='cuda', generator=g) + 0.5
    shift = torch.randn(cout, device='cuda', generator=g) * 0.1
    wp = w.permute(2, 3, 1, 0).contiguous().view(9, cin, cout)
    out = torch.zeros(B, H, W, cout, device='cuda', dtype=torch.float16)
    x_cl = _nhwc(x)
    rc = _lib.load().biu_conv_direct(ESZ_FP16, _lib.ptr(x_cl), cin, 0, cin, B, 1, H, W, 1, 3, 3, _lib.ptr(wp), cout,
                                     _lib.ptr(scale), _lib.ptr(shift), 0.1, _lib.ptr(out), cout, 0, _lib.stream_ptr())
    _lib.check(rc, 'biu_conv_direct')
    _sync_check()
    s, a = _layer_ref.conv_sums(_nhwc(x), w, 2)
    lo, hi = _layer_ref.interval(s, a, scale, shift, 0.1, 'fp16', _layer_ref.C_GPU)
    _layer_ref.check_interval(out.float(), lo, hi, 'conv_direct fp16')


@pytest.mark.parametrize('dims,mode', [(2, 0), (3, 0), (3, 1)])
def test_pool2_fp16(dims, mode):
    g = torch.Generator(device='cuda').manual_seed(19)
    B, C, D, H, W = 2, 32, (4 if dims == 3 else 1), 8, 12
    x = torch.randn((B, C, D, H, W) if dims == 3 else (B, C, H, W), device='cuda', generator=g).half()
    out = torch.zeros((B, D // 2, H // 2, W // 2, C) if dims == 3 else (B, H // 2, W // 2, C), device='cuda',
                      dtype=torch.float16)
    x_cl = _nhwc(x)
    rc = _lib.load().biu_pool2(ESZ_FP16, _lib.ptr(x_cl), C, 0, C, B, D, H, W, dims, mode, _lib.ptr(out), C, 0,
                               _lib.stream_ptr())
    _lib.check(rc, 'biu_pool2')
    _sync_check()
    if mode == 0:
        ref = (F.max_pool3d if dims == 3 else F.max_pool2d)(x, 2, 2)
    else:
        ref = F.interpolate(x, scale_factor=0.5, mode='nearest')
    assert torch.equal(_nchw(out), ref)
