"""The single-op interval check of tests/_layer_ref.py has teeth: an fp32-accumulated emulation of a layer passes it,
and each of the small kernel mistakes it is meant to catch fails it. Runs without a GPU."""
import math

import numpy as np
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


# ------------------------------------------------------------------------------------------------ Siam_UNet joins
def _twin_buffer(fmt, images, h=4, w=4, c=16, seed=5):
    g = torch.Generator().manual_seed(seed)
    return _operands(fmt, (images, h, w, c), g)


@pytest.mark.parametrize('shared', [0, 2])
def test_max_join_reference_and_planted_mistakes(shared):
    """The engine's stream addressing (net.cu stream_img0) passes; a stream taken one image off, and min in place of
    max, fail."""
    B = 3
    emb = _twin_buffer('bf16', B + shared if shared else 2 * B)
    cur0 = shared if shared else 0
    prev0 = 0 if shared else B
    want = R.max_join(*R.siam_streams(emb, B, shared))
    assert torch.equal(torch.maximum(emb[cur0:cur0 + B], emb[prev0:prev0 + B]), want)
    off = cur0 - 1 if shared else cur0 + 1          # current stream addressed one image off
    assert not torch.equal(torch.maximum(emb[off:off + B], emb[prev0:prev0 + B]), want)
    assert not torch.equal(torch.minimum(emb[cur0:cur0 + B], emb[prev0:prev0 + B]), want)


def _xcorr_emulate(cur, prev, fmt, near_pad=False, drop=None, trunc=False):
    """xcorr_join_kernel: out[b, y, x, c] = sum over i, j of cur[b, y + i - pt, x + j - pl, c] * prev[b, i, j, c],
    pt = (h - 1) // 2, pl = (w - 1) // 2, the in-bounds taps one after the other (i outer, j inner) with one fp32
    rounding each (fmaf), then one rounding to the storage format. near_pad: pt = h // 2, pl = w // 2 (the extra pad
    at the near end); drop = (i, j): that tap is left out; trunc: bf16 by truncation instead of rounding."""
    b, h, w, c = cur.shape
    pt, pl = (h // 2, w // 2) if near_pad else ((h - 1) // 2, (w - 1) // 2)
    xp = torch.nn.functional.pad(cur.double(), (0, 0, pl, w - 1 - pl, pt, h - 1 - pt))
    acc = torch.zeros(b, h, w, c, dtype=torch.float32)
    for i in range(h):
        for j in range(w):
            if (i, j) == drop:
                continue
            p = xp[:, i:i + h, j:j + w, :] * prev[:, i:i + 1, j:j + 1, :].double()   # exact products
            acc = (acc.double() + p).float()                                         # one rounding per tap
    if trunc:
        return (acc.view(torch.int32) & ~0xFFFF).view(torch.float32)
    return R.round_to(acc, fmt)


def _xcorr_check(got, cur, prev, fmt):
    s, a, n = R.xcorr_sums(cur, prev)
    lo, hi = R.xcorr_interval(s, a, n, fmt)
    R.check_interval(got, lo, hi, f'xcorr {fmt}')


@pytest.mark.parametrize('fmt', ['bf16', 'fp16', 'tf32', 'fp32'])
@pytest.mark.parametrize('hw', [(4, 4), (5, 3), (6, 8)])
def test_xcorr_reference_passes_the_kernel_emulation(fmt, hw):
    h, w = hw
    g = torch.Generator().manual_seed(h * 10 + w)
    op = 'bf16' if fmt == 'fp32' else fmt
    cur, prev = _operands(op, (2, h, w, 16), g), _operands(op, (2, h, w, 16), g)
    _xcorr_check(_xcorr_emulate(cur, prev, fmt), cur, prev, fmt)
    _, _, n = R.xcorr_sums(cur, prev)
    # 'same' padding with the extra pad at the far end: for even extents the near corner sees more taps than the far
    pt, pl = (h - 1) // 2, (w - 1) // 2
    assert float(n.max()) == h * w
    assert float(n[0, 0, 0, 0]) == (h - pt) * (w - pl) and float(n[0, -1, -1, 0]) == (pt + 1) * (pl + 1)


@pytest.mark.parametrize('mistake', ['near_pad', 'drop_border_tap', 'swap', 'bf16_trunc'])
def test_xcorr_reference_rejects_planted_mistakes(mistake):
    fmt = 'bf16'
    g = torch.Generator().manual_seed(9)
    cur, prev = _operands(fmt, (2, 4, 6, 16), g), _operands(fmt, (2, 4, 6, 16), g)
    if mistake == 'near_pad':              # even extents: the extra pad at the near end
        got = _xcorr_emulate(cur, prev, fmt, near_pad=True)
    elif mistake == 'drop_border_tap':     # the last tap of the correlation window left out
        got = _xcorr_emulate(cur, prev, fmt, drop=(3, 5))
    elif mistake == 'swap':                # cur and prev exchanged
        got = _xcorr_emulate(prev, cur, fmt)
    else:
        got = _xcorr_emulate(cur, prev, fmt, trunc=True)
    with pytest.raises(R.IntervalError):
        _xcorr_check(got, cur, prev, fmt)


def test_xcorr_reference_sees_one_dropped_tap_at_1024_taps():
    """32 x 32 embeddings: every output sums up to 1024 taps, the allowance is gamma_1024 A, and one dropped product
    still moves many outputs past it (tf32 storage, where no bf16 rounding hides the difference)."""
    g = torch.Generator().manual_seed(4)
    cur = _operands('tf32', (1, 32, 32, 4), g).abs()
    prev = _operands('tf32', (1, 32, 32, 4), g).abs()
    _xcorr_check(_xcorr_emulate(cur, prev, 'tf32'), cur, prev, 'tf32')
    with pytest.raises(R.IntervalError):
        _xcorr_check(_xcorr_emulate(cur, prev, 'tf32', drop=(16, 16)), cur, prev, 'tf32')


# ------------------------------------------------------------------------------------------------ bilinear x2
def test_bilinear_coordinates_match_pytorch_and_share_pairs():
    """For every extent 1 ... 64: the kernel's fp32 coordinate rule gives bit for bit the weights of PyTorch's float32
    F.interpolate(bilinear, align_corners=True), its (i0, i1) agree with the exact rule floor(o (n - 1) / (2n - 1)),
    and output rows 2p - 1 and 2p always interpolate between the same two source rows p - 1 and p. So
    up_bilinear_kernel's 2 x 2 path covers every output, and its per-pixel path is never taken."""
    f = torch.nn.functional
    for n in range(1, 65):
        x = torch.eye(n, dtype=torch.float32).reshape(1, n, n, 1)          # channel c: one-hot source row c
        y = f.interpolate(x, scale_factor=2, mode='bilinear', align_corners=True)[0, :, :, 0].t()
        assert torch.equal(y.double(), R._lerp_matrix(n, 'cpu')), n
        i0, i1, _ = R.bilinear_coord(n)
        o = torch.arange(2 * n, dtype=torch.int64)
        exact = torch.clamp((o * (n - 1)) // max(2 * n - 1, 1), max=n - 1)
        assert torch.equal(i0, exact) and torch.equal(i1, torch.clamp(exact + 1, max=n - 1)), n
        for p in range(1, n):
            assert int(i0[2 * p - 1]) == int(i0[2 * p]) == p - 1 and int(i1[2 * p - 1]) == int(i1[2 * p]) == p, (n, p)


def _bilinear_emulate(x, shift_src=False, copy_last_row=False):
    """up_bilinear_kernel in fp32: coordinates f = fp32((n-1)/(2n-1)) * o, lerps h0 (w0 v00 + w1 v01) + h1 (...),
    each product and sum rounded to fp32. shift_src: every source coordinate one pixel further (clamped);
    copy_last_row: the last output row is a copy of the row before."""
    def coords(n):
        s = np.float32(n - 1) / np.float32(2 * n - 1)
        out = []
        for o in range(2 * n):
            fo = np.float32(s * np.float32(o))
            i0 = min(int(fo), n - 1)
            l1 = np.float32(min(max(fo - np.float32(i0), np.float32(0)), np.float32(1)))
            if shift_src:
                i0 = min(i0 + 1, n - 1)
            out.append((i0, min(i0 + 1, n - 1), float(np.float32(1) - l1), float(l1)))
        return out
    b, h, w, c = x.shape
    ys, xs = coords(h), coords(w)
    xf = x.float()
    out = torch.empty(b, 2 * h, 2 * w, c, dtype=torch.float32)
    for oy, (y0, y1, h0, h1) in enumerate(ys):
        for ox, (x0, x1, w0, w1) in enumerate(xs):
            t = xf[:, y0, x0] * w0 + xf[:, y0, x1] * w1
            bt = xf[:, y1, x0] * w0 + xf[:, y1, x1] * w1
            out[:, oy, ox] = t * h0 + bt * h1
    if copy_last_row:
        out[:, -1] = out[:, -2]
    return out


def _bilinear_check(got, x, fmt):
    s, a = R.bilinear_x2(x)
    z = torch.zeros(x.shape[-1])
    lo, hi = R.interval(s, a, z + 1.0, z, 1.0, fmt, c=16.0)
    R.check_interval(got, lo, hi, f'bilinear {fmt}')


@pytest.mark.parametrize('fmt', ['bf16', 'fp16', 'tf32', 'fp32'])
@pytest.mark.parametrize('hw', [(1, 2), (3, 5), (8, 12)])
def test_bilinear_reference_passes_the_kernel_emulation(fmt, hw):
    g = torch.Generator().manual_seed(hw[0] * 100 + hw[1])
    x = _operands('bf16' if fmt == 'fp32' else fmt, (2, *hw, 16), g)
    _bilinear_check(R.round_to(_bilinear_emulate(x), fmt), x, fmt)


@pytest.mark.parametrize('mistake', ['align_corners_false', 'source_off_by_one', 'last_row_copied'])
@pytest.mark.parametrize('fmt', ['bf16', 'tf32'])
def test_bilinear_reference_rejects_planted_mistakes(mistake, fmt):
    g = torch.Generator().manual_seed(2)
    x = _operands(fmt, (2, 6, 10, 16), g)
    if mistake == 'align_corners_false':
        got = torch.nn.functional.interpolate(x.movedim(-1, 1), scale_factor=2, mode='bilinear',
                                              align_corners=False).movedim(1, -1)
    elif mistake == 'source_off_by_one':
        got = _bilinear_emulate(x, shift_src=True)
    else:
        got = _bilinear_emulate(x, copy_last_row=True)
    with pytest.raises(R.IntervalError):
        _bilinear_check(R.round_to(got, fmt), x, fmt)
