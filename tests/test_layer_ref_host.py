"""The single-op interval check of tests/_layer_ref.py has teeth: an fp32-accumulated emulation of a layer passes it,
and each of the small kernel mistakes it is meant to catch fails it. Runs without a GPU."""
import math

import pytest
import torch

from tests import _layer_ref as R


def _fmt_dtype(fmt):
    return {'bf16': torch.bfloat16, 'fp16': torch.float16}.get(fmt)


def _operands(fmt, shape, gen, scale=1.0):
    """Random values exactly representable in the operand format."""
    return R.round_to(torch.randn(shape, generator=gen, dtype=torch.float64) * scale, fmt)


def _layer(fmt, B=2, H=34, W=130, cin=32, cout=16, seed=0):
    g = torch.Generator().manual_seed(seed)
    x = _operands(fmt, (B, H, W, cin), g)
    w = _operands(fmt, (cout, cin, 3, 3), g, scale=(2.0 / (9 * cin)) ** 0.5)
    scale = (torch.rand(cout, generator=g) + 0.5).float()
    shift = (torch.randn(cout, generator=g) * 0.1).float()
    return x, w, scale, shift


def _emulate(x, w, scale, shift, slope, fmt, drop=None, extra_chunk=None):
    """Layer as a tensor-core kernel computes it: exact products of the operands, one fp32 addition at a time in
    (chunk of 16 channels, tap, channel) order, then fmaf(acc, scale, shift), LeakyReLU and one rounding.
    drop = (image, y, x, co, dy, dx, ci): leave that one product out; extra_chunk = k: add channel chunk k twice."""
    B, H, W, cin = x.shape
    cout = w.shape[0]
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1, 1, 1))
    acc = torch.zeros(B, H, W, cout, dtype=torch.float32)
    chunks = list(range(0, cin, 16)) + ([16 * extra_chunk] if extra_chunk is not None else [])
    for c0 in chunks:
        for dy in range(3):
            for dx in range(3):
                win = xp[:, dy:dy + H, dx:dx + W, :]
                for ci in range(c0, c0 + 16):
                    p = win[..., ci:ci + 1] * w[:, ci, dy, dx]            # exact in fp32
                    if drop is not None and (dy, dx, ci) == drop[4:]:
                        b, y, xx, co = drop[:4]
                        p[b, y, xx, co] = 0.0
                    acc = acc + p
    a = (acc.double() * scale.double() + shift.double()).float()
    return R.round_to(R.epilogue_fp32(a, slope), fmt)


def _interval(x, w, scale, shift, slope, fmt):
    """The interval with the allowance the GPU tests use (R.C_GPU), so the corruptions below fail at that width."""
    s, a = R.conv_sums(x, w, 2)
    return R.interval(s, a, scale, shift, slope, fmt, R.C_GPU)


@pytest.mark.parametrize('fmt', ['bf16', 'fp16', 'tf32'])
def test_fp32_accumulated_emulation_passes(fmt):
    x, w, scale, shift = _layer(fmt)
    got = _emulate(x, w, scale, shift, 0.1, fmt)
    s, a = R.conv_sums(x, w, 2)
    lo, hi = R.interval(s, a, scale, shift, 0.1, fmt, R.C_ACC)
    R.check_interval(got, lo, hi, f'emulated layer {fmt}')
    # for most elements the interval is a single stored value
    assert float((lo == hi).float().mean()) > 0.9


@pytest.mark.parametrize('dims,cin,fmt', [(2, 512, 'bf16'), (2, 512, 'fp32'), (3, 96, 'fp16'), (3, 96, 'fp32')])
def test_allowance_covers_cpu_float32_conv_at_the_largest_reductions(dims, cin, fmt):
    """C_ACC is the smallest power of two for which oneDNN's float32 convolution passes at K = 9 * 512 and 27 * 96
    (fp32 storage is the strictest case: no storage rounding hides the accumulation error)."""
    g = torch.Generator().manual_seed(3)
    spatial = (6, 10, 12) if dims == 3 else (16, 20)
    op = 'bf16' if fmt == 'fp32' else fmt
    x = _operands(op, (2, *spatial, cin), g)
    w = _operands(op, (32, cin) + (3,) * dims, g, scale=(2.0 / (cin * 3 ** dims)) ** 0.5)
    scale = (torch.rand(32, generator=g) + 0.5).float()
    shift = (torch.randn(32, generator=g) * 0.1).float()
    f = torch.nn.functional
    acc = (f.conv3d if dims == 3 else f.conv2d)(x.movedim(-1, 1), w, padding=1).movedim(1, -1)
    a = (acc.double() * scale.double() + shift.double()).float()
    got = R.round_to(R.epilogue_fp32(a, 0.1), fmt)
    s, aa = R.conv_sums(x, w, dims)
    c = R.min_c(got, s, aa, scale, shift, 0.1, fmt)
    assert c <= R.C_ACC, c


def _assert_fails(got, x, w, scale, shift, slope, fmt, what):
    lo, hi = _interval(x, w, scale, shift, slope, fmt)
    with pytest.raises(R.IntervalError):
        R.check_interval(got, lo, hi, what)


def _largest_product(x, w, b, y, xx, co):
    """(dy, dx, ci) of the largest |x * w| term of output (b, y, xx, co)."""
    xp = torch.nn.functional.pad(x, (0, 0, 1, 1, 1, 1))
    win = xp[b, y:y + 3, xx:xx + 3, :]                    # (3, 3, cin)
    t = (win * w[co].permute(1, 2, 0)).abs()
    k = int(torch.argmax(t))
    dy, rem = divmod(k, 3 * x.shape[-1])
    dx, ci = divmod(rem, x.shape[-1])
    return dy, dx, ci


@pytest.mark.parametrize('col', [127, 128])
def test_one_tap_dropped_at_a_strip_edge_fails(col):
    fmt = 'bf16'
    x, w, scale, shift = _layer(fmt)
    tap = _largest_product(x, w, 1, 5, col, 3)
    got = _emulate(x, w, scale, shift, 0.1, fmt, drop=(1, 5, col, 3) + tap)
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, f'tap dropped at x={col}')


def test_input_row_shifted_at_a_row_block_edge_fails():
    fmt = 'bf16'
    x, w, scale, shift = _layer(fmt)
    xs = x.clone()
    xs[:, 32] = x[:, 31]                 # the first row of the second 32-row block reads its predecessor
    got = _emulate(x, w, scale, shift, 0.1, fmt)
    got[:, 31:34] = _emulate(xs, w, scale, shift, 0.1, fmt)[:, 31:34]
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, 'row shifted')


@pytest.mark.parametrize('fmt', ['bf16', 'fp16'])
def test_truncation_instead_of_round_to_nearest_even_fails(fmt):
    x, w, scale, shift = _layer(fmt)
    a = _emulate(x, w, scale, shift, 0.1, 'fp32')
    u = a.view(torch.int32)
    if fmt == 'bf16':
        got = (u & ~0xFFFF).view(torch.float32)
    else:
        r = a.to(torch.float16).float()                 # round to nearest, then step towards zero where it rounded up
        up = r.abs() > a.abs()
        got = torch.where(up, torch.nextafter(r.to(torch.float16), torch.zeros_like(r, dtype=torch.float16)).float(), r)
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, f'{fmt} truncation')


@pytest.mark.parametrize('fmt', ['bf16', 'fp16', 'tf32'])
def test_one_ulp_bias_fails(fmt):
    x, w, scale, shift = _layer(fmt)
    got = _emulate(x, w, scale, shift, 0.1, fmt)
    if fmt == 'tf32':
        got = (got.view(torch.int32) + 0x2000).view(torch.float32)
    else:
        dt = _fmt_dtype(fmt)
        got = torch.nextafter(got.to(dt), torch.full_like(got, math.inf, dtype=dt)).float()
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, 'one-ulp bias')


def test_two_channel_scales_swapped_fails():
    fmt = 'fp16'
    x, w, scale, shift = _layer(fmt)
    sw = scale.clone()
    sw[[4, 5]] = scale[[5, 4]]
    got = _emulate(x, w, sw, shift, 0.1, fmt)
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, 'scales swapped')


def test_k_split_group_counted_twice_fails():
    fmt = 'bf16'
    x, w, scale, shift = _layer(fmt, H=8, W=20)
    got = _emulate(x, w, scale, shift, 0.1, fmt, extra_chunk=1)
    _assert_fails(got, x, w, scale, shift, 0.1, fmt, 'K chunk twice')


@pytest.mark.parametrize('dims', [2, 3])
def test_pool_one_pixel_off_fails(dims):
    g = torch.Generator().manual_seed(4)
    shape = (2, 8, 12, 16) if dims == 2 else (2, 4, 8, 12, 16)
    x = R.round_to(torch.randn(shape, generator=g), 'bf16')
    assert torch.equal(R.maxpool(x, dims), R.maxpool(x.clone(), dims))
    off = torch.roll(x, 1, dims=dims)                  # every window one column to the left
    assert not torch.equal(R.maxpool(off, dims), R.maxpool(x, dims))


def test_rounding_modes_match_the_host_packers():
    # bf16: nearest even; 1 + 2^-8 is a tie between 1 and 1 + 2^-7
    v = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8)], dtype=torch.float64)
    assert R.round_to(v, 'bf16').tolist() == [1.0, 1 + 2 ** -6, -1.0]
    # tf32: ties away from zero (cvt.rna); 1 + 2^-11 is a tie between 1 and 1 + 2^-10
    v = torch.tensor([1 + 2 ** -11, -(1 + 2 ** -11), 1 + 2 ** -12], dtype=torch.float64)
    assert R.round_to(v, 'tf32').tolist() == [1 + 2 ** -10, -(1 + 2 ** -10), 1.0]
    # fp16: nearest even, beyond 65504 (from 65520 on) +-inf
    v = torch.tensor([1 + 2 ** -11, 65519.0, 65520.0, -70000.0], dtype=torch.float64)
    assert R.round_to(v, 'fp16').tolist() == [1.0, 65504.0, math.inf, -math.inf]


def test_interval_keeps_infinities_of_fp16_overflow():
    s = torch.tensor([60000.0, 70000.0, -70000.0, 1.0], dtype=torch.float64)
    lo, hi = R.interval(s, s.abs(), torch.ones(1), torch.zeros(1), 1.0, 'fp16')
    got = torch.tensor([60000.0, math.inf, -math.inf, 1.0])
    R.check_interval(got, lo, hi, 'overflow')
    with pytest.raises(R.IntervalError):
        R.check_interval(torch.tensor([60000.0, 65504.0, -math.inf, 1.0]), lo, hi, 'saturated')
