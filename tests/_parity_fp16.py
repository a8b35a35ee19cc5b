"""Parity gate of the fp16 mode: the reference's own float16 arithmetic on the same weights and input.

Mirrors the bf16 yardstick of oracle/yardstick.py and tests/_parity.py with float16:

* ``autocast_fp16(fn, ...)``  - the oracle forward under ``torch.autocast(dtype=torch.float16)`` (the reference's
  ``model.half()`` arithmetic with fp32 BatchNorm statistics);
* ``operand_rounded_fp16(fn, ...)`` - the oracle forward in fp32 with the two operands of every convolution rounded to
  float16 first (fp32 accumulation and BatchNorm): the arithmetic of an F16 tensor-core GEMM with an fp32 epilogue.

The yardstick is the larger of the two errors against the plain fp32 oracle run, as for bf16. ``extend_parity``
teaches tests/_parity.py's bound functions the precision name 'fp16', so that the parity tests written for every
precision (they take it as a parameter and ask tests/_parity.py for the bound) hold the fp16 mode to this yardstick.
"""
import contextlib

import torch

from oracle import yardstick as ys
from tests import _parity

NORTH_STAR = 1e-3        # default init: the tf32 gate (fp16 keeps tf32's 10 mantissa bits)


def round_fp16(t):
    """Round-to-nearest-even to float16 (beyond +-65504: +-inf, as a float16 store does)."""
    return t.to(torch.float16).to(torch.float32)


def operand_rounded_fp16(fn, *args, **kwargs):
    """fn(*args) with every convolution's input and weight rounded to float16, fp32 accumulate."""
    with torch.no_grad(), ys._RoundConvOperands(round_fp16):
        return fn(*args, **kwargs)


def autocast_fp16(fn, *args, **kwargs):
    """fn(*args) under torch.autocast(float16) on the device of the first tensor argument."""
    dev = next((a.device.type for a in args if torch.is_tensor(a)), 'cpu')
    with torch.no_grad(), torch.autocast(dev, dtype=torch.float16):
        return fn(*args, **kwargs)


def _runs(fn, *args):
    return [ys._first(autocast_fp16(fn, *args)), ys._first(operand_rounded_fp16(fn, *args))]


def yardstick(fn, *args, ref=None):
    """max |fp16 reference - fp32 reference|: the larger of the autocast run and the operand-rounded emulation."""
    with torch.no_grad():
        if ref is None:
            ref = ys._first(fn(*args))
        return max((r - ref).abs().max().item() for r in _runs(fn, *args))


def errors(fn, *args, ref=None):
    """(max, mean) abs error of the reference's fp16 arithmetic against its fp32 run."""
    with torch.no_grad():
        if ref is None:
            ref = ys._first(fn(*args))
        d = [(r - ref).abs() for r in _runs(fn, *args)]
    return max(x.max().item() for x in d), max(x.mean().item() for x in d)


def per_channel_bound(fn, *args, ref=None):
    """(C,) tensor: bound on the max-abs error of every output channel (tests/_parity.py per_channel_bound, fp16)."""
    with torch.no_grad():
        if ref is None:
            ref = ys._first(fn(*args))
        red = [d for d in range(ref.dim()) if d != 1]
        scale = ref.abs().amax(dim=red).clamp(min=1.0)
        yard = torch.stack([(r - ref).abs().amax(dim=red) for r in _runs(fn, *args)]).amax(0)
    return _parity.YARD_FACTOR * yard + _parity.FLOOR * scale


@contextlib.contextmanager
def extend_parity():
    """Within the block, tests/_parity.py answers precision 'fp16' with the fp16 yardstick (every other precision
    exactly as before)."""
    errors0, per_channel0 = _parity.errors, _parity.per_channel_bound

    def errors_any(fn, precision, *args, ref=None):
        return errors(fn, *args, ref=ref) if precision == 'fp16' else errors0(fn, precision, *args, ref=ref)

    def per_channel_any(fn, precision, *args, ref=None):
        return per_channel_bound(fn, *args, ref=ref) if precision == 'fp16' else per_channel0(fn, precision, *args, ref=ref)

    _parity.errors, _parity.per_channel_bound = errors_any, per_channel_any
    _parity.NORTH_STAR['fp16'] = NORTH_STAR
    try:
        yield
    finally:
        _parity.errors, _parity.per_channel_bound = errors0, per_channel0
        del _parity.NORTH_STAR['fp16']
