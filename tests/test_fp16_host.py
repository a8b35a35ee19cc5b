"""Host-side checks of the fp16 precision mode (no GPU): its yardstick, its name in the precision table, and the range
of the stress nets the fp16 GPU tests run (fp16 stores do not saturate: a value beyond 65504 would become inf on the
device, so those tests must not come near it)."""
import numpy as np
import pytest
import torch
from torch.overrides import TorchFunctionMode

from oracle import models as omodels
from oracle import yardstick as ys
from tests import _golden, _parity, _parity_fp16
from tests import test_gpu_baseline_sizes as sizes
from tests import test_gpu_unet as unet

FP16_HEADROOM = 65504.0 / 16


def test_fp16_yardstick_lies_between_tf32_and_bf16():
    tiles = torch.randint(0, 256, (2, 1, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(22))
    sd = unet.stress_state_dict(8, 22)
    x = tiles.float() / 255
    y = {p: ys.yardstick(omodels.unet_forward, p, sd, x) for p in ('tf32', 'bf16')}
    y['fp16'] = _parity_fp16.yardstick(omodels.unet_forward, sd, x)
    assert y['tf32'] <= y['fp16'] <= y['bf16'], y


def test_extend_parity_answers_fp16_only():
    tiles = torch.randint(0, 256, (1, 1, 32, 32), dtype=torch.uint8, generator=torch.Generator().manual_seed(4))
    sd, x = unet.stress_state_dict(4, 4), tiles.float() / 255
    before = {p: _parity.bound(omodels.unet_forward, p, sd, x) for p in ('fp32', 'tf32', 'bf16')}
    with _parity_fp16.extend_parity():
        assert {p: _parity.bound(omodels.unet_forward, p, sd, x) for p in ('fp32', 'tf32', 'bf16')} == before
        mx, mean = _parity_fp16.errors(omodels.unet_forward, sd, x)
        assert _parity.bound(omodels.unet_forward, 'fp16', sd, x) == (_parity.YARD_FACTOR * mx + _parity.FLOOR,
                                                                      _parity.YARD_FACTOR * mean + _parity.FLOOR)
        assert _parity.NORTH_STAR['fp16'] == 1e-3
    assert 'fp16' not in _parity.NORTH_STAR


def test_round_fp16_is_round_to_nearest_even():
    t = torch.tensor([1.0 + 2 ** -11, 1.0 + 3 * 2 ** -11, 65504.0, 65520.0, -1e5])
    assert _parity_fp16.round_fp16(t).tolist() == [1.0, 1.0 + 2 ** -9, 65504.0, float('inf'), float('-inf')]


def test_unknown_precision_lists_fp16():
    from bio_image_unet_b200.engine import PRECISION, Engine
    assert PRECISION['fp16'] == 3                # BIU_PREC_FP16 (include/biu_b200.h)
    with pytest.raises(ValueError, match="'fp16'"):
        Engine('unet2d', {}, 8, precision='fp8')


class _MaxAbs(TorchFunctionMode):
    """Largest |value| of every floating-point tensor a torch function returns during a forward."""

    def __init__(self):
        super().__init__()
        self.max = 0.0

    def __torch_function__(self, func, types, args=(), kwargs=None):
        out = func(*args, **(kwargs or {}))
        for t in (out if isinstance(out, (tuple, list)) else (out,)):
            if torch.is_tensor(t) and t.is_floating_point() and t.numel():
                self.max = max(self.max, t.detach().abs().max().item())
        return out


def _max_activation(fn, *args):
    with torch.no_grad(), _MaxAbs() as m:
        fn(*args)
    return m.max


def _unet3d_cfg4_net():
    """The stress UNet3D(16) of the cfg-4 test (tests/test_gpu_baseline_sizes.py), on a crop of its patch."""
    from bio_image_unet_b200.unet3d import UNet3D
    g = torch.Generator().manual_seed(41)
    x_u8 = torch.randint(0, 256, (32, 1, 64, 128, 128), dtype=torch.uint8, generator=g)
    torch.manual_seed(2)
    sd = sizes._stress_module_sd(UNet3D(n_filter=16), 41)
    x = x_u8[:1, :, :16, :64, :64].float() / 255
    with torch.no_grad():
        _, lg = omodels.unet3d_forward(sd, x[:1, :, :16, :32, :32])
    return sizes._unit_logits(sd, lg, 'final.weight', 'final.bias'), x


@pytest.mark.parametrize('net', ['fp16_vs_bf16', 'cta_pairs', 'fused_pool', 'cfg2', 'cfg4', 'golden_unet', 'golden_unet3d'])
def test_stress_nets_stay_far_below_fp16_range(net):
    if net == 'fp16_vs_bf16':
        tiles = torch.randint(0, 256, (2, 1, 128, 128), dtype=torch.uint8, generator=torch.Generator().manual_seed(8))
        fn, args = omodels.unet_forward, (unet.unit_logit_state_dict(32, 132, tiles), tiles.float() / 255)
    elif net == 'cta_pairs':
        x = torch.randint(0, 256, (6, 1, 128, 128), dtype=torch.uint8, generator=torch.Generator().manual_seed(12))
        fn, args = omodels.unet_forward, (unet.unit_logit_state_dict(32, 55, x), x[:2].float() / 255)
    elif net == 'fused_pool':
        x = torch.randint(0, 256, (3, 1, 64, 64), dtype=torch.uint8, generator=torch.Generator().manual_seed(3))
        fn, args = omodels.unet_forward, (unet.stress_state_dict(32, seed=9), x.float() / 255)
    elif net == 'cfg2':
        probe = torch.randint(0, 256, (1, 1, 512, 512), dtype=torch.uint8, generator=torch.Generator().manual_seed(5))
        fn, args = omodels.unet_forward, (unet.unit_logit_state_dict(32, 302, probe), probe.float() / 255)
    elif net == 'cfg4':
        fn, args = omodels.unet3d_forward, _unet3d_cfg4_net()
    elif net == 'golden_unet':
        g = _golden.load('unet_single')
        fn, args = omodels.unet_forward, (_golden.state_dict(g), torch.from_numpy(np.ascontiguousarray(g['patches'])).float() / 255)
    else:
        g = _golden.load('unet3d_overlap')
        fn = omodels.unet3d_forward
        args = (_golden.state_dict(g), torch.from_numpy(np.ascontiguousarray(g['patches'][:2])).float()[:, None] / 255)
    m = _max_activation(fn, *args)
    assert 0 < m < FP16_HEADROOM, (net, m)
