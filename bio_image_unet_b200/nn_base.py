"""Shared plumbing of the model classes: the reference's ``nn.Module`` surface (constructor arguments, parameter
names / shapes, ``forward`` return convention) on top of the B200 engine.

* ``model.eval()`` + CUDA input  -> engine (tcgen05 kernels through the C-ABI);
* ``model.train()``              -> plain PyTorch ops (training itself is outside this engine's scope, the path
                                    exists so checkpoints can be produced with the same classes);
* ``model.eval()`` + CPU input   -> RuntimeError: there is deliberately no CPU inference fallback.
"""
import torch
from torch import nn

from .engine import Engine


def conv_block(dims, in_channels, out_channels, kernel_size=3, dropout=0., dilation=1):
    """Conv -> BatchNorm -> LeakyReLU(0.1) -> Dropout, registered as '<name>.0' / '<name>.1' like
    unet/unet.py:54-60 and unet3d/unet3d.py:52-58 (state_dict compatibility)."""
    conv, bn, drop = (nn.Conv2d, nn.BatchNorm2d, nn.Dropout2d) if dims == 2 else (nn.Conv3d, nn.BatchNorm3d, nn.Dropout3d)
    return nn.Sequential(conv(in_channels, out_channels, kernel_size, padding=dilation, dilation=dilation),
                         bn(out_channels), nn.LeakyReLU(negative_slope=0.1, inplace=True), drop(dropout))


class EngineModule(nn.Module):
    """Base class: lazily builds / rebuilds an Engine from the current parameters."""

    precision = 'tf32'          # engine-only knob: 'tf32' | 'fp16' | 'bf16' | 'fp32' (see unet.Predict)

    def _engine_spec(self):     # -> dict(kind=..., n_filter=..., in_channels=..., heads=[...], ...)
        raise NotImplementedError

    def _signature(self):
        return tuple((t.data_ptr(), t._version) for t in list(self.parameters()) + list(self.buffers())) + (self.precision,)

    def _get_engine(self, device, raw_logits):
        key = (self._signature(), str(device), raw_logits)
        cache = self.__dict__.setdefault('_engine_cache', {})
        if cache.get('key') != key:
            if cache.get('engine') is not None:
                cache['engine'].close()
            spec = self._engine_spec()
            if raw_logits:
                spec['heads'] = [(n, c, None) for n, c, _ in spec['heads']]
            cache['engine'] = Engine(state_dict=self.state_dict(), precision=self.precision, device=device, **spec)
            cache['key'] = key
            cache['plan'] = None
        return cache['engine'], cache

    def _engine_forward(self, x, prev=None, raw_logits=True):
        if not x.is_cuda:
            raise RuntimeError(f'{type(self).__name__}: eval-mode forward needs CUDA tensors '
                               '(bio_image_unet_b200 has no CPU inference fallback)')
        eng, cache = self._get_engine(x.device, raw_logits)
        plan = (x.shape[0], tuple(x.shape[2:]))
        if cache['plan'] != plan:
            eng.plan(x.shape[0], tuple(x.shape[2:]))
            cache['plan'] = plan
        x = x.to(torch.float32).contiguous()
        prev = None if prev is None else prev.to(torch.float32).contiguous()
        val, _ = eng.forward(x, prev, want_val=True, want_u8=False)
        return val
