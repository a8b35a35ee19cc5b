"""Parity of the 2D U-Net path on the GPU: engine forward vs the CPU oracle, and the whole Predict pipeline vs
the golden fixtures produced by the unmodified reference.

Tolerances (BASELINE.json north_star): fp32/TF32 mode max-abs 1e-3 on the sigmoid output, bf16 mode 1e-2 - asserted on
PyTorch's default random init; on stress-initialised nets the reduced-precision modes are held to 1.5x the error of
the reference's own arithmetic at that precision on the same weights and input (tests/_parity.py, oracle/yardstick.py).
Tile indices, uint8 tiles and the stitch are bit-exact.
"""
import os

import numpy as np
import pytest
import torch

from oracle import models as omodels
from oracle import pipeline as opipe
from tests import _golden, _parity

pytestmark = pytest.mark.gpu

# Stated tolerances (max-abs on the sigmoid output) - gate on PyTorch's default random init:
TOL = _parity.NORTH_STAR
# "Stress" regime (Kaiming weights, randomised BN statistics, logits rescaled to unit variance: every pixel sits on
# the steep part of the sigmoid): no constants - _parity.check / _parity.bound compare with the reference's own
# reduced-precision arithmetic on the same weights (measured there: TF32 operand rounding 1.3e-3 .. 3.1e-3, bf16
# autocast 1.3e-2 .. 2.7e-2 on these nets, growing with the number of pixels the maximum is taken over).


def golden_lsb(forward, precision, sd, patches):
    """Allowance on the uint8-quantised result tiles of a golden fixture, in LSB: 1 (truncation) + 1.5 x what the
    reference's arithmetic at that precision moves the sigmoid on the fixture's own weights and tiles."""
    x = torch.from_numpy(np.ascontiguousarray(patches)).float() / 255
    return _parity.lsb_bound(forward, precision, sd, x)


def stress_state_dict(n_filter, seed, head_gain=4.0):
    """Kaiming conv weights + randomised BatchNorm statistics (SURVEY.md §7.2), built on the product's own class."""
    from bio_image_unet_b200.unet import Unet
    g = torch.Generator().manual_seed(seed)
    m = Unet(n_filter=n_filter)
    sd = m.state_dict()
    for k, v in sd.items():
        if k.endswith('num_batches_tracked'):
            continue
        if k.endswith('.0.weight') or (k.startswith('up') and k.endswith('weight')):
            fan_in = v[0].numel() if not k.startswith('up') else v.shape[0]
            sd[k] = torch.randn(v.shape, generator=g) * (2.0 / 1.01 / fan_in) ** 0.5
            if k.startswith('final'):
                sd[k] *= head_gain
        elif k.endswith('.0.bias') or (k.startswith('up') and k.endswith('bias')):
            sd[k] = torch.randn(v.shape, generator=g) * 0.05
        elif k.endswith('running_var') or k.endswith('.1.weight'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
    return sd


def unit_logit_state_dict(n_filter, seed, tiles):
    """Stress init with the head rescaled so that the oracle's logits have zero mean / unit variance."""
    sd = stress_state_dict(n_filter, seed, head_gain=1.0)
    with torch.no_grad():
        _, lg = omodels.unet_forward(sd, tiles.float() / 255)
    sd['final.0.weight'] = sd['final.0.weight'] / lg.std()
    sd['final.0.bias'] = (sd['final.0.bias'] - lg.mean()) / lg.std()
    return sd


def default_state_dict(n_filter, seed):
    from bio_image_unet_b200.unet import Unet
    torch.manual_seed(seed)
    return Unet(n_filter=n_filter).state_dict()


@pytest.mark.parametrize('precision', ['fp32', 'tf32', 'bf16'])
@pytest.mark.parametrize('regime', ['default', 'stress'])
@pytest.mark.parametrize('n_filter,tile,batch', [(4, (32, 48), 3), (32, (64, 64), 2), (16, (128, 32), 1)])
def test_engine_forward_matches_oracle(precision, regime, n_filter, tile, batch):
    from bio_image_unet_b200.engine import Engine
    g = torch.Generator().manual_seed(7)
    tiles = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=g)
    if regime == 'default':
        sd = default_state_dict(n_filter, seed=100 + n_filter)
    else:
        sd = unit_logit_state_dict(n_filter, 100 + n_filter, tiles)
    x = tiles.float() / 255
    with torch.no_grad():
        ref, _ = omodels.unet_forward(sd, x)
    eng = Engine('unet2d', sd, n_filter, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
    eng.plan(batch, tile)
    val, u8 = eng.forward(tiles.cuda(), want_val=True, want_u8=True)
    torch.cuda.synchronize()
    err, _, tol = _parity.check(val, ref, omodels.unet_forward, precision, sd, x, what=f'unet nf={n_filter} {regime}')
    if regime == 'default':
        assert err < TOL[precision], (precision, regime, err)
    # quantised output: trunc(sigmoid*255) within 1 LSB of the oracle's (+ the float tolerance in LSBs)
    ref_u8 = (ref.numpy() * 255).astype('uint8')
    d = np.abs(u8.cpu().numpy().astype(np.int16) - ref_u8.astype(np.int16))
    assert d.max() <= 1 + int(np.ceil(tol * 255)), d.max()
    if regime == 'default':
        mask_ref, mask = ref > 0.5, val.cpu() > 0.5
        union = (mask_ref | mask).sum().item()
        iou = (mask_ref & mask).sum().item() / union if union else 1.0
        assert iou >= 0.999, iou
    eng.close()


@pytest.mark.parametrize('precision', ['tf32', 'bf16'])
def test_bimodal_mask_iou(precision):
    """Decisive-output regime: logits scaled by 60 so that |logit| >> rounding noise for most pixels. A random net
    has Gaussian logits, i.e. always some pixels arbitrarily close to the decision boundary where ANY reduced
    precision flips the mask (the reference's own bf16 autocast reaches IoU 0.988 on such a net, SURVEY.md §7.2);
    a trained net is bimodal. So: thresholded-mask IoU >= 0.999 (north_star) over the pixels whose reference logit
    is decisive (|logit| above the mode's noise floor), plus the stated max-abs tolerance on those pixels."""
    from bio_image_unet_b200.engine import Engine
    g = torch.Generator().manual_seed(11)
    tiles = torch.randint(0, 256, (2, 1, 128, 128), dtype=torch.uint8, generator=g)
    sd = unit_logit_state_dict(32, 77, tiles)
    sd['final.0.weight'] = sd['final.0.weight'] * 60
    sd['final.0.bias'] = sd['final.0.bias'] * 60
    with torch.no_grad():
        ref, logits = omodels.unet_forward(sd, tiles.float() / 255)
    eng = Engine('unet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
    eng.plan(2, (128, 128))
    val, _ = eng.forward(tiles.cuda(), want_val=True)
    val = val.cpu()
    decided = logits.abs() > (12 if precision == 'bf16' else 8)      # logit sigma is 60 here
    assert decided.float().mean() > 0.8
    mask_ref, mask = (ref > 0.5) & decided, (val > 0.5) & decided
    iou = (mask_ref & mask).sum().item() / max((mask_ref | mask).sum().item(), 1)
    assert iou >= 0.999, iou
    assert (val - ref).abs()[decided].max().item() < TOL[precision]
    iou_all = ((ref > 0.5) & (val > 0.5)).sum().item() / max(((ref > 0.5) | (val > 0.5)).sum().item(), 1)
    assert iou_all >= (0.99 if precision == 'bf16' else 0.998), iou_all
    eng.close()


def test_engine_tensor_path_matches_cuda_core_path():
    """Same weights, tf32 storage: tcgen05 kernels vs the direct CUDA-core kernels on intermediate activations (cat4, mid2, d7).
    Both paths store tf32-representable float32 values (low 13 mantissa bits zero); the 'fp32' mode does not round."""
    from bio_image_unet_b200.engine import Engine
    sd = stress_state_dict(32, seed=5)
    tiles = torch.randint(0, 256, (2, 1, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(1)).cuda()
    acts = [('d7', 32, 0), ('cat4', 64, 0), ('mid2', 512, 4)]
    eng = Engine('unet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision='tf32', device='cuda:0')
    eng.plan(2, (64, 64))
    v_tc, _ = eng.forward(tiles, want_val=True)
    a_tc = {n: eng.debug_activation(n, c, l) for n, c, l in acts}
    eng.set_force_direct(1)
    eng.plan(2, (64, 64))
    v_dc, _ = eng.forward(tiles, want_val=True)
    a_dc = {n: eng.debug_activation(n, c, l) for n, c, l in acts}
    eng.close()
    for n in a_tc:   # both paths round every stored activation to tf32; only the accumulation order differs
        rel = np.abs(a_tc[n] - a_dc[n]).max() / np.abs(a_dc[n]).max()
        assert rel < 1e-2, (n, rel)
        for path, a in (('tcgen05', a_tc[n]), ('cuda-core', a_dc[n])):
            assert not (a.view(np.uint32) & 0x1FFF).any(), (n, path, 'stores a value that is not tf32-representable')
    assert (v_tc - v_dc).abs().max().item() < 5e-2   # stress net, logit sigma ~13
    eng = Engine('unet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision='fp32', device='cuda:0')
    eng.plan(2, (64, 64))
    eng.forward(tiles, want_val=True)
    for n, c, l in acts:
        assert (eng.debug_activation(n, c, l).view(np.uint32) & 0x1FFF).any(), (n, 'fp32 mode rounded every value to tf32')
    eng.close()


@pytest.mark.parametrize('name', ['unet_single', 'unet_all_invert', 'unet_first_u8', 'unet_small_reflect'])
@pytest.mark.parametrize('precision', ['fp32', 'tf32', 'bf16'])
def test_predict_matches_reference_golden(name, precision, tmp_path):
    from bio_image_unet_b200 import tiff
    from bio_image_unet_b200.unet import Predict
    g = _golden.load(name)
    ckpt = str(tmp_path / 'model.pt')
    torch.save({'state_dict': _golden.state_dict(g), 'n_filter': int(g['n_filter']), 'in_channels': 1,
                'out_channels': 1}, ckpt)
    imgs = g['imgs'].copy()
    res_file = str(tmp_path / 'res.tif')
    p = Predict(imgs, res_file, ckpt, network='Unet', resize_dim=tuple(int(v) for v in g['resize_dim']),
                invert=bool(g['invert']), normalization_mode=str(g['mode']), clip_threshold=tuple(g['clip']),
                add_tile=int(g['add_tile']), show_progress=False, device='cuda:0', precision=precision,
                keep_intermediates=True)
    # indices: bit-exact
    assert (p.N_x, p.N_y) == (int(g['N_x']), int(g['N_y']))
    assert np.array_equal(p.X_start, g['X_start']) and np.array_equal(p.Y_start, g['Y_start'])
    assert p.X_start.dtype == np.uint16
    # normalisation + split: bit-exact uint8 tiles; 'single' overwrites the caller's array like the reference
    assert np.array_equal(p.patches, g['patches'])
    if str(g['mode']) == 'single':
        assert np.array_equal(imgs, g['imgs_after'])
    # forward: quantised result tiles within 1 LSB (+ 1.5 x the reference's own reduced-precision error)
    lsb = golden_lsb(omodels.unet_forward, precision, _golden.state_dict(g), g['patches'])
    d = np.abs(p.result_patches.astype(np.int16) - g['result_patches'].astype(np.int16))
    assert d.max() <= lsb, d.max()
    # stitch: bit-exact given the engine's own tiles
    grid = (p.N_x, p.N_y, p.X_start, p.Y_start)
    st = opipe.stitch_mean_2d(p.result_patches, g['imgs'].shape[0], g['imgs'].shape[1:],
                              tuple(int(v) for v in g['resize_dim']), grid)
    out = tiff.imread(res_file)
    assert out.dtype == np.float16 and out.shape == g['result_file'].shape
    assert np.array_equal(out, st.astype('float16'))
    assert np.abs(out.astype(np.float32) - g['result_file'].astype(np.float32)).max() <= lsb


def test_normalisation_kernels_bit_exact():
    from bio_image_unet_b200 import engine as E
    rng = np.random.default_rng(3)
    for dtype, hi in (('uint16', 4096), ('uint16', 65536), ('uint8', 256)):
        for clip in ((0., 99.8), (0.5, 99.98), (2., 100.)):
            for invert in (False, True):
                stack = rng.integers(0, hi, (3, 37, 53)).astype(dtype)
                stack[1] = (rng.normal(300, 40, (37, 53)).clip(0, hi - 1)).astype(dtype)
                ref = opipe.preprocess_stack(stack.copy(), 'single', clip, invert).astype('uint8')
                dev = torch.from_numpy(stack).cuda()
                hist = E.histogram(dev)
                assert np.array_equal(hist[0].cpu().numpy(), np.bincount(stack[0].ravel(), minlength=65536))
                lut, params = E.norm_lut(hist, hist, 3, clip[0], clip[1], invert)
                got = E.apply_lut(dev, lut).cpu().numpy()
                assert np.array_equal(got, ref), (dtype, hi, clip, invert)
                lo_ref = np.nanpercentile(stack[2], clip[0]); hi_ref = np.percentile(stack[2], clip[1])
                assert params[2, 0].item() == lo_ref and params[2, 1].item() == hi_ref


@pytest.mark.parametrize('dtype', ['uint16', 'uint8'])
def test_fused_normalise_gather_equals_two_pass(dtype):
    """biu_gather_tiles_lut (normalisation fused into the split: what Session.predict_device and the 3D sessions run)
    against biu_apply_lut + biu_gather_tiles and against the oracle's preprocess + split: bit-exact, per-frame and
    stack-wide tables, reflect / zero padding of undersized frames, 16-pixel vector and 4-pixel scalar runs."""
    from bio_image_unet_b200 import engine as E
    from bio_image_unet_b200 import tiling
    rng = np.random.default_rng(12)
    hi = 4096 if dtype == 'uint16' else 256
    for (f, h, w, th, tw, add, pad_mode) in [(3, 80, 112, 32, 48, 1, 0), (2, 40, 40, 64, 64, 0, 0), (2, 40, 40, 64, 64, 0, 1),
                                              (4, 64, 96, 32, 24, 2, 0), (1, 96, 160, 32, 160, 0, 0)]:
        stack = rng.integers(0, hi, (f, h, w)).astype(dtype)
        dev = torch.from_numpy(stack).cuda()
        hist = E.histogram(dev)
        n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
        for per_frame in (True, False):
            if per_frame:
                lut, _ = E.norm_lut(hist, hist, f, 0.5, 99.5, False)
            else:
                tot = E.hist_sum(hist)
                lut, _ = E.norm_lut(tot, tot, 1, 0.5, 99.5, False)
            two = E.gather_tiles(E.apply_lut(dev, lut).view(f, 1, h, w), [0], xs, ys, (1, th, tw), pad_mode)
            one = E.gather_tiles_lut(dev.view(f, 1, h, w), lut, [0], xs, ys, (1, th, tw), pad_mode)
            assert torch.equal(one, two), (dtype, f, h, w, th, tw, add, pad_mode, per_frame)
        if pad_mode == 0 and dtype == 'uint16':          # and against the reference's numpy path ('single' mode)
            lut, _ = E.norm_lut(hist, hist, f, 0.0, 99.8, False)
            one = E.gather_tiles_lut(dev.view(f, 1, h, w), lut, [0], xs, ys, (1, th, tw), 0)
            want = opipe.split_2d(opipe.preprocess_stack(stack.copy(), 'single', (0., 99.8), False), (th, tw), add)[0]
            assert np.array_equal(one.cpu().numpy().reshape(want.shape), want)


def test_stitch_mean_bit_exact():
    from bio_image_unet_b200 import engine as E
    from bio_image_unet_b200 import tiling
    rng = np.random.default_rng(4)
    # (96, 200, ..., add 14): more than eight tiles cover a 16-pixel run (the kernel's list of covering columns overflows
    # and it walks all columns); (64, 256, 32, 64): aligned 16-byte vector loads and stores
    for (h, w, th, tw, add, c) in [(70, 90, 32, 48, 1, 1), (64, 64, 32, 32, 2, 2), (20, 100, 32, 48, 0, 1), (33, 47, 16, 16, 3, 1),
                                   (96, 200, 32, 160, 14, 1), (64, 256, 32, 64, 1, 2)]:
        n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
        f = 2
        tiles = rng.integers(0, 256, (f * n_x * n_y, c, th, tw)).astype('uint8')
        ref = opipe.stitch_mean_2d(tiles, f, (h, w), (th, tw), (n_x, n_y, xs, ys)).reshape(f, c, h, w)
        got = E.stitch_mean_u8(torch.from_numpy(tiles).cuda(), f, c, (h, w), xs, ys, (th, tw)).cpu().numpy()
        assert np.array_equal(got, ref)


@pytest.mark.parametrize('precision', ['tf32', 'bf16'])
@pytest.mark.parametrize('tile', [(64, 64), (48, 80), (128, 32)])
def test_fused_maxpool_is_bit_identical(precision, tile):
    """MaxPool2d(2) fused into the preceding block's epilogue (warp shuffles over the stored values) vs the
    standalone pool kernel: pooled tensors m1..m4 and the network output must be bit-identical."""
    from bio_image_unet_b200.engine import Engine
    sd = stress_state_dict(32, seed=9)
    tiles = torch.randint(0, 256, (3, 1, *tile), dtype=torch.uint8, generator=torch.Generator().manual_seed(3)).cuda()
    eng = Engine('unet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
    eng.plan(3, tile)
    names = [('m1', 32, 1), ('m2', 64, 2), ('m3', 128, 3), ('m4', 256, 4)]
    v_fused, u_fused = eng.forward(tiles, want_val=True)
    a_fused = {n: eng.debug_activation(n, c, l).copy() for n, c, l in names}
    eng.set_fuse_pool(0)
    eng.workspace.zero_()
    v_plain, u_plain = eng.forward(tiles, want_val=True)
    a_plain = {n: eng.debug_activation(n, c, l).copy() for n, c, l in names}
    for n, _, _ in names:
        assert np.array_equal(a_fused[n], a_plain[n]), n
    assert torch.equal(v_fused, v_plain) and torch.equal(u_fused, u_plain)
    eng.close()


# ---------------------------------------------------------------------------------------------------------------
# AttentionUnet / Unet_v0 (unet.Predict(network=...), unet/predict.py:89-97)
# ---------------------------------------------------------------------------------------------------------------
def _variant_state_dict(network, n_filter, seed, stress):
    """State dict of the product's own module class; 'stress' = Kaiming weights + randomised BN statistics."""
    from bio_image_unet_b200.unet import AttentionUnet, Unet_v0
    torch.manual_seed(seed)
    m = (AttentionUnet if network == 'AttentionUnet' else Unet_v0)(n_filter=n_filter)
    sd = m.state_dict()
    if not stress:
        return sd
    g = torch.Generator().manual_seed(seed)
    for k, v in sd.items():
        if k.endswith('num_batches_tracked'):
            continue
        if k.endswith('.0.weight') or (k.startswith('up') and k.endswith('weight')):
            fan_in = v[0].numel() if not k.startswith('up') else v.shape[0]
            sd[k] = torch.randn(v.shape, generator=g) * (2.0 / fan_in) ** 0.5
        elif k.endswith('.0.bias') or (k.startswith('up') and k.endswith('bias')):
            sd[k] = torch.randn(v.shape, generator=g) * 0.05
        elif k.endswith('running_var') or k.endswith('.1.weight'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        else:
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
    return sd


@pytest.mark.parametrize('precision', ['fp32', 'tf32', 'bf16'])
@pytest.mark.parametrize('regime', ['default', 'stress'])
@pytest.mark.parametrize('network,n_filter,tile,batch', [('AttentionUnet', 32, (64, 64), 2), ('AttentionUnet', 8, (32, 48), 3),
                                                         ('AttentionUnet', 16, (256, 128), 1),
                                                         ('Unet_v0', 32, (64, 64), 2), ('Unet_v0', 4, (48, 32), 3),
                                                         ('Unet_v0', 16, (256, 128), 1)])
def test_variant_forward_matches_oracle(precision, regime, network, n_filter, tile, batch):
    from bio_image_unet_b200.engine import Engine
    g = torch.Generator().manual_seed(17)
    tiles = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=g)
    sd = _variant_state_dict(network, n_filter, 200 + n_filter, regime == 'stress')
    forward = omodels.FORWARD_2D[network]
    with torch.no_grad():
        ref, logits = forward(sd, tiles.float() / 255)
        if regime == 'stress':          # rescale the head so that the logits have unit variance (steep sigmoid)
            sd['final.0.weight'] = sd['final.0.weight'] / logits.std()
            sd['final.0.bias'] = (sd['final.0.bias'] - logits.mean()) / logits.std()
            ref, logits = forward(sd, tiles.float() / 255)
    kind = 'attunet2d' if network == 'AttentionUnet' else 'unet2d_v0'
    eng = Engine(kind, sd, n_filter, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
    eng.plan(batch, tile)
    val, u8 = eng.forward(tiles.cuda(), want_val=True, want_u8=True)
    torch.cuda.synchronize()
    err, _, tol = _parity.check(val, ref, forward, precision, sd, tiles.float() / 255, what=f'{network} nf={n_filter} {regime}')
    if regime == 'default':
        assert err < TOL[precision], (network, precision, regime, err)
    ref_u8 = (ref.numpy() * 255).astype('uint8')
    d = np.abs(u8.cpu().numpy().astype(np.int16) - ref_u8.astype(np.int16))
    assert d.max() <= 1 + int(np.ceil(tol * 255)), d.max()
    eng.close()


def test_attention_gate_matches_oracle_activations():
    """The gated skip tensors a1..a4 (skip * psi) against the oracle, exact-fp32 mode and tf32 tensor-core mode."""
    from bio_image_unet_b200.engine import Engine
    sd = _variant_state_dict('AttentionUnet', 32, 5, True)
    tiles = torch.randint(0, 256, (2, 1, 128, 128), dtype=torch.uint8, generator=torch.Generator().manual_seed(2))
    acts = {}
    with torch.no_grad():
        omodels.attention_unet_forward(sd, tiles.float() / 255, collect=acts)
    for precision, tol in (('fp32', 2e-4), ('tf32', 3e-2)):
        eng = Engine('attunet2d', sd, 32, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
        eng.plan(2, (128, 128))
        eng.forward(tiles.cuda(), want_val=True)
        for k, (c, level) in enumerate([(256, 3), (128, 2), (64, 1), (32, 0)]):
            cat = eng.debug_activation(f'cat{k + 1}', 2 * c, level)          # [up | gated skip], NHWC
            got = torch.from_numpy(cat[:, 0, :, :, c:].copy()).permute(0, 3, 1, 2)
            ref = acts[f'a{k + 1}']
            scale = ref.abs().max().item()
            assert (got - ref).abs().max().item() <= tol * max(scale, 1.0), (precision, k)
        eng.close()


@pytest.mark.parametrize('name', ['attunet_single', 'unetv0_all'])
@pytest.mark.parametrize('precision', ['fp32', 'tf32', 'bf16'])
@pytest.mark.parametrize('as_class', [False, True])
def test_variant_predict_matches_reference_golden(name, precision, as_class, tmp_path):
    from bio_image_unet_b200 import tiff, unet
    g = _golden.load(name)
    network = str(g['network'])
    params = {'state_dict': _golden.state_dict(g), 'n_filter': int(g['n_filter']), 'in_channels': 1, 'out_channels': 1}
    if network == 'Unet_v0':            # old checkpoints carry no channel counts (unet/predict.py:94-97)
        del params['in_channels'], params['out_channels']
    ckpt = str(tmp_path / 'model.pt')
    torch.save(params, ckpt)
    imgs = g['imgs'].copy()
    res_file = str(tmp_path / 'res.tif')
    net_arg = getattr(unet, network) if as_class else network
    p = unet.Predict(imgs, res_file, ckpt, network=net_arg, resize_dim=tuple(int(v) for v in g['resize_dim']),
                     invert=bool(g['invert']), normalization_mode=str(g['mode']), clip_threshold=tuple(g['clip']),
                     add_tile=int(g['add_tile']), show_progress=False, device='cuda:0', precision=precision,
                     keep_intermediates=True)
    assert (p.N_x, p.N_y) == (int(g['N_x']), int(g['N_y']))
    assert np.array_equal(p.X_start, g['X_start']) and np.array_equal(p.Y_start, g['Y_start'])
    assert np.array_equal(p.patches, g['patches'])
    lsb = golden_lsb(omodels.FORWARD_2D[network], precision, _golden.state_dict(g), g['patches'])
    d = np.abs(p.result_patches.astype(np.int16) - g['result_patches'].astype(np.int16))
    assert d.max() <= lsb, (d.max(), lsb)
    out = tiff.imread(res_file)
    assert out.dtype == np.float16 and out.shape == g['result_file'].shape
    assert np.abs(out.astype(np.float32) - g['result_file'].astype(np.float32)).max() <= lsb


# ---------------------------------------------------------------------------------------------------------------
# Row-streaming folded-tap kernel (conv_rows.cuh): narrow 3x3 blocks on planes at least 128 pixels wide
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture
def rows_kernel_toggle():
    from bio_image_unet_b200 import _lib
    lib = _lib.load()
    yield lambda on: lib.biu_set_rows_kernel(int(on))   # 0: halo kernel, 1: row kernel, 2: row kernel, both pipelines forced
    lib.biu_set_rows_kernel(1)


@pytest.mark.parametrize('precision', ['tf32', 'bf16'])
@pytest.mark.parametrize('n_filter,tile,batch', [(32, (64, 256), 2), (32, (48, 144), 3), (16, (80, 128), 2), (32, (16, 640), 1),
                                                 (32, (80, 400), 1)])
def test_rows_kernel_matches_halo_kernel_2d(precision, n_filter, tile, batch, rows_kernel_toggle):
    """Same network, narrow blocks (encode2 + fused pool, decode7, decode8 + head) through conv_rows vs conv_halo:
    identical up to the fp32 summation order of the three partial rows (one ulp of the stored format), and both
    within tolerance of the oracle. W = 144 / 640 exercise a partial last strip, H = 48 / 80 / 16 partial row blocks;
    (80, 400) puts the 64-channel blocks of level 1 (200 px wide: a partial second strip) and decode5's channel-chunk
    slots on ragged extents."""
    from bio_image_unet_b200.engine import Engine
    sd = stress_state_dict(n_filter, seed=21)
    tiles = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=torch.Generator().manual_seed(4))
    sd = unit_logit_state_dict(n_filter, 21, tiles)
    with torch.no_grad():
        ref, _ = omodels.unet_forward(sd, tiles.float() / 255)
    names = [('cat4', 2 * n_filter, 0), ('m1', n_filter, 1), ('d7', n_filter, 0)]
    got = {}
    for on in (2, 1, 0):                  # 2: both pipelines of the row kernel forced on (default only for big batches)
        rows_kernel_toggle(on)
        eng = Engine('unet2d', sd, n_filter, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
        eng.plan(batch, tile)
        val, u8 = eng.forward(tiles.cuda(), want_val=True, want_u8=True)
        got[on] = (val.cpu(), u8.cpu(), {n: eng.debug_activation(n, c, l).copy() for n, c, l in names})
        eng.close()
    # one or two pipelines: the same MMAs in the same order per output row -> bit-identical
    assert torch.equal(got[2][0], got[1][0]) and torch.equal(got[2][1], got[1][1])
    for n, _, _ in names:
        assert np.array_equal(got[2][2][n], got[1][2][n]), n
    rel = 2 ** -7 if precision == 'bf16' else 2 ** -9       # one ulp of the stored format
    for n, _, _ in names:
        a, b = got[1][2][n], got[0][2][n]
        if n == 'cat4':                   # [up4 | encode2]: only the skip half comes straight out of a narrow block
            a, b = a[..., n_filter:], b[..., n_filter:]
        # encode2 / m1 come straight out of the first narrow block; d7 has the whole network in between
        assert np.abs(a - b).max() <= (8 if n == 'd7' else 1) * rel * max(np.abs(b).max(), 1.0), \
            (n, np.abs(a - b).max(), np.abs(b).max())
    x = tiles.float() / 255
    _, _, tol = _parity.check(got[1][0], ref, omodels.unet_forward, precision, sd, x, what='row kernel')
    _parity.check(got[0][0], ref, omodels.unet_forward, precision, sd, x, what='halo kernel')
    # the two kernels round every stored activation independently: their difference is of the size of the error itself
    assert (got[1][0] - got[0][0]).abs().max().item() < tol
    assert np.abs(got[1][1].numpy().astype(np.int16) - got[0][1].numpy().astype(np.int16)).max() <= \
        1 + int(np.ceil(tol * 255))


@pytest.mark.parametrize('precision', ['tf32', 'bf16'])
@pytest.mark.parametrize('kind,n_filter,tile,batch', [('unet3d', 16, (8, 16, 128), 2), ('unet3d', 32, (16, 24, 128), 1),
                                                      ('mo3d', 16, (8, 32, 256), 1),
                                                      # planes narrower than 128 px: the row kernel's PLANE mode (16 x 8 tiles,
                                                      # dz folded into N, planes streamed); W = 40 / H = 48: ragged tiles
                                                      ('unet3d', 16, (16, 32, 64), 2), ('unet3d', 32, (16, 48, 40), 1),
                                                      ('mo3d', 16, (16, 32, 96), 1), ('unet3d', 16, (32, 64, 64), 3)])
def test_rows_kernel_matches_halo_kernel_3d(precision, kind, n_filter, tile, batch, rows_kernel_toggle):
    from bio_image_unet_b200.engine import Engine
    from bio_image_unet_b200.multi_output_unet3d import MultiOutputUnet3D
    from bio_image_unet_b200.unet3d import UNet3D
    torch.manual_seed(31)
    if kind == 'unet3d':
        module, heads = UNet3D(n_filter=n_filter), [('', 1, 'sigmoid')]
        spec = dict(n_filter=n_filter, in_channels=1, heads=heads)
    else:
        cfg = {'seg': {'channels': 1, 'activation': 'sigmoid'}, 'flow': {'channels': 2, 'activation': None}}
        module = MultiOutputUnet3D(1, cfg, n_filter, True)
        spec = dict(n_filter=n_filter, in_channels=1, heads=[('seg', 1, 'sigmoid'), ('flow', 2, None)], use_interpolation=True)
    sd = module.state_dict()
    g = torch.Generator().manual_seed(8)
    for k, v in sd.items():                       # randomised BN statistics so that the folding is exercised
        if k.endswith('running_var') or k.endswith('.1.weight'):
            sd[k] = torch.rand(v.shape, generator=g) + 0.5
        elif k.endswith('running_mean') or k.endswith('.1.bias'):
            sd[k] = torch.randn(v.shape, generator=g) * 0.1
    x = torch.rand((batch, 1, *tile), generator=g)
    if kind == 'unet3d':
        fwd = lambda sd_, x_: omodels.unet3d_forward(sd_, x_)[0]                       # noqa: E731
    else:
        def fwd(sd_, x_):
            o = omodels.mo3d_forward(sd_, x_, cfg, True)
            return torch.cat([o['seg'].float(), o['flow'].float()], 1)
    with torch.no_grad():
        ref = fwd(sd, x)
    got = {}
    for on in (2, 1, 0):                  # 2: both pipelines of the row kernel forced on
        rows_kernel_toggle(on)
        eng = Engine(kind, sd, precision=precision, device='cuda:0', **spec)
        eng.plan(batch, tile)
        val, _ = eng.forward(x.cuda(), want_val=True, want_u8=False)
        got[on] = val.cpu()
        eng.close()
    assert torch.equal(got[2], got[1])    # one or two pipelines: bit-identical
    _, _, tol = _parity.check(got[1], ref, fwd, precision, sd, x, what=f'{kind} row kernel')
    _parity.check(got[0], ref, fwd, precision, sd, x, what=f'{kind} halo kernel')
    assert (got[1] - got[0]).abs().max().item() < tol


@pytest.mark.parametrize('name', ['unet_f32_single', 'unet_f32_first_invert', 'unet_f32_all'])
@pytest.mark.parametrize('precision', ['fp32', 'bf16'])
def test_predict_float32_stack_matches_reference_golden(name, precision, tmp_path):
    """float32 input stacks: percentiles by exact radix select on the device, the reference's float32 arithmetic;
    uint8 tiles bit-exact, 'single' mode writes the float32 normalised frames back into the caller's array."""
    from bio_image_unet_b200 import tiff
    from bio_image_unet_b200.unet import Predict
    g = _golden.load(name)
    ckpt = str(tmp_path / 'model.pt')
    torch.save({'state_dict': _golden.state_dict(g), 'n_filter': int(g['n_filter']), 'in_channels': 1,
                'out_channels': 1}, ckpt)
    imgs = g['imgs'].copy()
    assert imgs.dtype == np.float32
    res_file = str(tmp_path / 'res.tif')
    p = Predict(imgs, res_file, ckpt, network='Unet', resize_dim=tuple(int(v) for v in g['resize_dim']),
                invert=bool(g['invert']), normalization_mode=str(g['mode']), clip_threshold=tuple(float(v) for v in g['clip']),
                add_tile=int(g['add_tile']), show_progress=False, device='cuda:0', precision=precision,
                keep_intermediates=True)
    assert np.array_equal(p.patches, g['patches'])
    if str(g['mode']) == 'single':
        assert np.array_equal(imgs, g['imgs_after'])
    else:
        assert np.array_equal(imgs, g['imgs'])
    d = np.abs(p.result_patches.astype(np.int16) - g['result_patches'].astype(np.int16))
    lsb = golden_lsb(omodels.unet_forward, precision, _golden.state_dict(g), g['patches'])
    assert d.max() <= lsb, (d.max(), lsb)
    out = tiff.imread(res_file)
    assert out.shape == g['result_file'].shape and out.dtype == np.float16


def test_float32_normalisation_kernel_bit_exact():
    """biu_normalize_f32 against numpy on awkward float data: negatives, denormal-ish magnitudes, ties, constant rows."""
    from bio_image_unet_b200 import engine as E
    rng = np.random.default_rng(5)
    for mode in ('single', 'first', 'all'):
        for invert in (False, True):
            stack = (rng.standard_normal((3, 37, 53)) * rng.choice([1e-3, 1.0, 4e4])).astype(np.float32)
            stack[1, :5] = stack[1, 0, 0]                     # ties
            stack[2] = np.round(stack[2], 1)
            ref = opipe.preprocess_stack(stack.copy(), mode, (0.5, 99.3), invert)
            u8, f32, _ = E.normalize_f32(torch.from_numpy(stack).cuda(), mode, 0.5, 99.3, invert, want_f32=True)
            # (a constant frame gives 0 / 0 = NaN in numpy and on the device alike)
            assert np.array_equal(f32.cpu().numpy(), ref.astype(np.float32), equal_nan=True), (mode, invert)
            ok = ~np.isnan(ref)
            assert np.array_equal(u8.cpu().numpy()[ok], ref.astype(np.float32)[ok].astype(np.uint8)), (mode, invert)


# ---------------------------------------------------------------------------------------------------------------
# CTA pairs in the halo-tile kernel (tcgen05.mma.cta_group::2, conv_halo.cuh)
# ---------------------------------------------------------------------------------------------------------------
@pytest.fixture
def cta2_toggle():
    from bio_image_unet_b200 import _lib
    lib = _lib.load()
    yield lambda on: lib.biu_set_halo_cta2(int(on))
    lib.biu_set_halo_cta2(1)


@pytest.mark.parametrize('precision', ['bf16', 'tf32'])
@pytest.mark.parametrize('kind,n_filter,tile,batch', [('unet2d', 32, (128, 128), 6), ('unet2d', 32, (64, 96), 2), ('unet2d', 16, (256, 64), 3),
                                                      ('unet3d', 32, (16, 32, 32), 2)])
def test_cta_pairs_match_single_cta(precision, kind, n_filter, tile, batch, cta2_toggle):
    """Same network with the wide layers (>= 64 output channels per block) on CTA pairs (one MMA of M = 256 over two
    SMs, each CTA staging half of every weight tile) and on single CTAs: per output tile the same MMAs in the same
    order, so activations and outputs are bit-identical; and the paired run matches the oracle."""
    from bio_image_unet_b200.engine import Engine
    from bio_image_unet_b200.unet3d import UNet3D
    g = torch.Generator().manual_seed(12)
    x = torch.randint(0, 256, (batch, 1, *tile), dtype=torch.uint8, generator=g)
    if kind == 'unet2d':
        sd = unit_logit_state_dict(n_filter, 55, x)
        names = [('mid2', 16 * n_filter, 4), ('d2', 8 * n_filter, 3), ('d4', 4 * n_filter, 2), ('cat3', 4 * n_filter, 1)]
        fwd = omodels.unet_forward
    else:
        torch.manual_seed(7)
        sd = UNet3D(n_filter=n_filter).state_dict()
        names = []
        fwd = lambda sd_, x_: omodels.unet3d_forward(sd_, x_)                              # noqa: E731
    got = {}
    for on in (1, 0):
        cta2_toggle(on)
        eng = Engine(kind, sd, n_filter, 1, [('', 1, 'sigmoid')], precision=precision, device='cuda:0')
        eng.plan(batch, tile)
        val, u8 = eng.forward(x.cuda(), want_val=True, want_u8=True)
        torch.cuda.synchronize()
        got[on] = (val.cpu(), u8.cpu(), {n: eng.debug_activation(n, c, l).copy() for n, c, l in names})
        assert eng.fallback_ops == 0
        eng.close()
    for n, _, _ in names:
        assert np.array_equal(got[1][2][n], got[0][2][n]), n
    assert torch.equal(got[1][0], got[0][0]) and torch.equal(got[1][1], got[0][1])
    xf = x.float() / 255
    with torch.no_grad():
        ref = fwd(sd, xf)[0]
    _parity.check(got[1][0], ref, fwd, precision, sd, xf, what=f'{kind} CTA pairs')
