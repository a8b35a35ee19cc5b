"""Exact single-op reference of the engine's layer program, and the interval check built on it.

Every tensor-core op of the engine is "fp32 accumulation of exactly representable operands, an fp32 epilogue, one
rounding to the storage format". So each op can be recomputed from the engine's OWN stored input in float64, and the
engine's stored output is required to be the correctly rounded value, up to an allowance for the fp32 accumulation:

    S = exact conv of the stored input with the rounded weights       (float64)
    A = conv of |input| with |weights|                                (float64)
    d = C * 2^-24 * A                                                 (accumulation allowance, in units of S)
    stored output in [round_F(epi(S - d)), round_F(epi(S + d))]        (epi: the monotone fp32 epilogue)

epi(s) = max(a, a * slope) with a = fmaf(s, scale, shift); both ends are evaluated like the kernels do, in fp32, so
for most elements the interval is ONE value: a wrong rounding mode, a one-ulp bias, a missing tap or a wrong
scale / shift index fails it. Nothing compounds from layer to layer, and no yardstick is involved.

Parameter folding mirrors net_finalize (bio_image_unet_b200/csrc/net.cu):
  - BatchNorm in float64, cast to fp32: scale = g / sqrt(var + 1e-5), shift = beta + (bias - mean) * scale.
  - Tensor-core ops: weights rounded to the operand format (bf16 / fp16: round to nearest even; tf32: round to
    nearest, ties away, as host_round_tf32 and cvt.rna do); the scale is applied in the fp32 epilogue.
  - CUDA-core ops (fp32 mode, the +16 fallback, the first block of the 3D nets): the checkpoint's fp32 weights as
    they are (w_direct), fp32 fmaf accumulation, and the same fmaf(acc, scale, shift) epilogue; the BatchNorm scale is
    not folded into these weights.
  - First block of the 2D nets on the row kernel (first mode): raw uint8 values times the rounded weights, with
    scale_first = fp32(scale) / 255.0f.
  - Attention gate: the BatchNorm scales are inside the weights (fp32(sc * w), then rounded for the tensor cores),
    scale 1.
  - Transposed conv: scale 1, shift = bias.

Works on CPU and CUDA tensors alike (the GPU tests compute their references in float64 on the device).
"""
import math
import warnings

import torch

FORMATS = ('bf16', 'fp16', 'tf32', 'fp32')

# Smallest power of two for which a CPU float32 convolution (oneDNN's summation order) passes the check at the
# largest reductions the suite uses, 9 * 512 (2D) and 27 * 96 (3D); see tests/test_layer_ref_host.py.
C_ACC = 4.0
# The kernels on the B200 need more. tcgen05 does not add one product at a time with round-to-nearest: with C_ACC about
# one stored value in a million lands one ulp short, always towards zero. Measured over tests/test_gpu_layer_exact.py,
# the tcgen05 ops need c = 16 in bf16 and fp16 and c = 32 in tf32. The CUDA-core kernels' fmaf chains with fp32
# storage also exceed C_ACC by one fp32 ulp in a few values out of 10^5. d = 2^-19 A then stays below a quarter of an
# fp16 ulp wherever |S| is more than A / 64.
C_GPU = 32.0


def pad16(c):
    return (c + 15) // 16 * 16


# ------------------------------------------------------------------------------------------------ rounding
def round_to(x, fmt):
    """Value of x (any float tensor) after it is computed in fp32 and stored in format fmt, as float32.
    bf16 / fp16: round to nearest even (fp16 beyond +-65504 becomes +-inf); tf32: round to nearest, ties away from
    zero (cvt.rna.tf32.f32); fp32: fp32 itself."""
    x = x.to(torch.float32)
    if fmt == 'bf16':
        return x.to(torch.bfloat16).to(torch.float32)
    if fmt == 'fp16':
        return x.to(torch.float16).to(torch.float32)
    if fmt == 'tf32':
        u = x.view(torch.int32)
        finite = (u & 0x7F800000) != 0x7F800000
        r = torch.where(finite, (u + 0x1000) & ~0x1FFF, u)
        return r.view(torch.float32)
    if fmt == 'fp32':
        return x
    raise ValueError(f'unknown format {fmt!r}')


def operand_format(precision):
    """Format of the tensor-core operands / stored activations of a precision mode."""
    return {'bf16': 'bf16', 'fp16': 'fp16', 'tf32': 'tf32', 'fp32': 'fp32'}[precision]


# ------------------------------------------------------------------------------------------------ folding
def fold_bn(sd, conv_key, bn_key):
    """(w fp32 (Cout, Cin, [kd,] kh, kw), scale fp32, shift fp32) of a Conv + BatchNorm block, as net_finalize."""
    w = sd[conv_key + '.weight'].detach().cpu().float()
    b = sd[conv_key + '.bias'].detach().cpu().double()
    g = sd[bn_key + '.weight'].detach().cpu().double()
    be = sd[bn_key + '.bias'].detach().cpu().double()
    mu = sd[bn_key + '.running_mean'].detach().cpu().double()
    var = sd[bn_key + '.running_var'].detach().cpu().double()
    s = g / torch.sqrt(var + 1e-5)
    return w, s.float(), (be + (b - mu) * s).float()


def fold_gate(sd, name, c):
    """AttentionBlock 'name' reading [gate (c) | skip (c)]: GEMM weights fp32(sc * w) (Cout, 2c), shift, and the psi
    head (weights, bias) with BatchNorm(1) folded, as net_finalize."""
    ws, shift = [], None
    for br in ('.W_gate', '.W_x'):
        w, s, sh = fold_bn(sd, name + br + '.0', name + br + '.1')
        w = w.reshape(w.shape[0], c).double()
        ws.append((s.double()[:, None] * w).float())
        shift = sh if shift is None else (shift + sh)       # fp32 sum, as the host's shift[co] += (float)...
    w, s, sh = fold_bn(sd, name + '.psi.0', name + '.psi.1')
    gw = (s.double() * w.reshape(-1).double()).float()
    return torch.cat(ws, 1), shift, gw, sh


# ------------------------------------------------------------------------------------------------ reference
def _conv(x, w, dims):
    """x (N, C, [D,] H, W), w (Cout, C, [kd,] kh, kw), both float64, zero padding 1."""
    f = torch.nn.functional
    return f.conv3d(x, w, padding=1) if dims == 3 else f.conv2d(x, w, padding=1)


def _cl_to_cf(x):       # (N, [D,] H, W, C) -> (N, C, [D,] H, W)
    return x.movedim(-1, 1)


def conv_sums(x, w, dims):
    """S and A of a 3x3(x3) convolution of a channels-last input x (N, [D,] H, W, Cin) with w (Cout, Cin, ...):
    channels-last float64 results (N, [D,] H, W, Cout)."""
    xd = _cl_to_cf(x.double())
    wd = w.double().to(xd.device)
    s = _conv(xd, wd, dims).movedim(1, -1)
    a = _conv(xd.abs(), wd.abs(), dims).movedim(1, -1)
    return s, a


def up_sums(x, w, dims):
    """Transposed conv, kernel 2 stride 2 (no bias): x (N, [D,] H, W, Cin), w (Cin, Cout, [2,] 2, 2)."""
    f = torch.nn.functional
    xd = _cl_to_cf(x.double())
    wd = w.double().to(xd.device)
    t = f.conv_transpose3d if dims == 3 else f.conv_transpose2d
    return t(xd, wd, stride=2).movedim(1, -1), t(xd.abs(), wd.abs(), stride=2).movedim(1, -1)


def gemm_sums(x, w):
    """1x1 conv: x (..., Cin), w (Cout, Cin)."""
    xd, wd = x.double(), w.double().to(x.device)
    return xd @ wd.t(), xd.abs() @ wd.abs().t()


def epilogue_fp32(a32, slope):
    """max(a, a * slope) in fp32: LeakyReLU for 0 <= slope <= 1 (1: identity, 0: ReLU)."""
    return torch.maximum(a32, a32 * torch.tensor(slope, dtype=torch.float32, device=a32.device))


def interval(s, a, scale, shift, slope, fmt, c=C_ACC):
    """[lo, hi] (float32) of the stored value of fmt(max(t, t * slope)), t = fmaf(s', scale, shift), over every fp32
    accumulation s' within c * 2^-24 * A of the exact sum S."""
    d = a * (c * 2.0 ** -24)
    sc = scale.double().to(s.device)
    sh = shift.double().to(s.device)
    e1 = (s - d) * sc + sh
    e2 = (s + d) * sc + sh
    lo, hi = torch.minimum(e1, e2), torch.maximum(e1, e2)
    lo = epilogue_fp32(lo.float(), slope)
    hi = epilogue_fp32(hi.float(), slope)
    return round_to(lo, fmt), round_to(hi, fmt)


def head_interval(vlo, vhi, hw, hb, act, rel=1e-5):
    """Bounds of act(sum_k hw[h, k] * v_k + hb[h]) for every v in the box [vlo, vhi] (..., K), with a relative
    allowance rel of sum |hw * v| + |hb| for the fp32 evaluation of the head. Returns (lo, hi) (..., heads)."""
    hw = hw.double().to(vlo.device)
    hb = hb.double().to(vlo.device)
    p1 = vlo.double()[..., None, :] * hw
    p2 = vhi.double()[..., None, :] * hw
    lo = torch.minimum(p1, p2).sum(-1) + hb
    hi = torch.maximum(p1, p2).sum(-1) + hb
    mag = torch.maximum(p1.abs(), p2.abs()).sum(-1) + hb.abs()
    lo, hi = lo - rel * mag, hi + rel * mag
    return activation(lo, act), activation(hi, act)


def activation(x, act):
    if act in (None, 'none'):
        return x
    if act == 'sigmoid':
        return torch.sigmoid(x)
    if act == 'tanh':
        return torch.tanh(x)
    if act == 'relu':
        return torch.relu(x)
    raise ValueError(act)


# ------------------------------------------------------------------------------------------------ check
class IntervalError(AssertionError):
    pass


def violations(got, lo, hi):
    """Boolean mask of the elements outside [lo, hi] (NaN is always outside)."""
    got = got.to(lo.device).float()
    return ~((got >= lo) & (got <= hi))


def check_interval(got, lo, hi, what, ref=None, index=None, atol=0.0):
    """Raise IntervalError naming the count and the worst element (its (image, [z,] y, x, channel)), got / ref /
    interval, when any stored value of got lies outside [lo - atol, hi + atol]."""
    got = got.to(lo.device).float()
    bad = violations(got, lo - atol, hi + atol)
    n = int(bad.sum())
    if n == 0:
        return
    dist = torch.where(bad, torch.maximum(lo - got, got - hi).nan_to_num(math.inf), torch.zeros_like(got))
    k = int(torch.argmax(dist.reshape(-1)))
    coord = list(torch.unravel_index(torch.tensor(k), got.shape))
    coord = [int(v) for v in coord]
    if index is not None:
        coord[0] = index[coord[0]]
    r = '' if ref is None else f' ref={float(ref.reshape(-1)[k]):.9g}'
    raise IntervalError(f'{what}: {n} of {got.numel()} values outside the interval; worst at (image, [z,] y, x, c)='
                        f'{tuple(coord)}: got={float(got.reshape(-1)[k]):.9g}{r} interval=['
                        f'{float(lo.reshape(-1)[k]):.9g}, {float(hi.reshape(-1)[k]):.9g}]')


def min_c(got, s, a, scale, shift, slope, fmt, ladder=(0.0, 0.25, 0.5, 1.0, 2.0, 4.0, 8.0, 16.0, 32.0, 64.0, 128.0,
                                                       256.0, 1024.0)):
    """Smallest c of the ladder for which every element passes (inf when none does): how much of the accumulation
    allowance an op actually needed."""
    got = got.to(s.device).float()
    for c in ladder:
        lo, hi = interval(s, a, scale, shift, slope, fmt, c)
        if not bool(violations(got, lo, hi).any()):
            return c
    return math.inf


def maxpool(x, dims):
    """2 x 2 (x 2) max pool of a channels-last tensor: bit-exact, as the kernels take a max of stored values."""
    if dims == 2:
        n, h, w, c = x.shape
        return x.reshape(n, h // 2, 2, w // 2, 2, c).amax((2, 4))
    n, d, h, w, c = x.shape
    return x.reshape(n, d // 2, 2, h // 2, 2, w // 2, 2, c).amax((2, 4, 6))


def trilinear_x2(x):
    """F.interpolate(scale_factor=2, mode='trilinear', align_corners=False) of (N, D, H, W, C) in float64, and the
    matching |.|-sum for the allowance (the weights are non-negative, so it is the same interpolation of |x|)."""
    f = torch.nn.functional
    xd = _cl_to_cf(x.double())
    r = f.interpolate(xd, scale_factor=2, mode='trilinear', align_corners=False).movedim(1, -1)
    a = f.interpolate(xd.abs(), scale_factor=2, mode='trilinear', align_corners=False).movedim(1, -1)
    return r, a


def nearest_x2(x, dims):
    if dims == 2:
        return x.repeat_interleave(2, 1).repeat_interleave(2, 2)
    return x.repeat_interleave(2, 1).repeat_interleave(2, 2).repeat_interleave(2, 3)


# ------------------------------------------------------------------------------------------------ Siam_UNet joins
def siam_streams(emb, batch, shared):
    """(current, previous) embeddings of a twin-encoder buffer emb (images, ..., C) as the engine addresses them
    (stream_img0 in net.cu): [current (B) | previous (B)], or with the shared encoder previous = images [0, B) and
    current = images [shared, shared + B)."""
    if shared > 0:
        return emb[shared:shared + batch], emb[:batch]
    return emb[:batch], emb[batch:2 * batch]


def max_join(cur, prev):
    """torch.maximum of the two stored embeddings: bit-exact, the kernel takes the maximum of stored values."""
    return torch.maximum(cur, prev)


def xcorr_sums(cur, prev):
    """Depth-wise cross-correlation of Siam_UNet mode='corr' (siam_unet.py:75-83) of channels-last embeddings cur, prev
    (B, h, w, C): S = F.conv2d(cur, prev, groups=B*C, padding='same') in float64 as PyTorch computes it (for even
    extents the extra padding is at the far end), A the same of |cur|, |prev|, and the number n of in-bounds taps of
    every output (a 'same' convolution of ones). Channels-last float64 (B, h, w, C) results; n (1, h, w, 1)."""
    f = torch.nn.functional
    b, h, w, c = cur.shape
    x = _cl_to_cf(cur.double()).reshape(1, b * c, h, w)
    k = _cl_to_cf(prev.double()).reshape(b * c, 1, h, w)
    one = torch.ones((1, 1, h, w), dtype=torch.float64, device=x.device)
    with warnings.catch_warnings():      # even extents: PyTorch notes that it pads a copy of the input
        warnings.simplefilter('ignore', UserWarning)
        s = f.conv2d(x, k, groups=b * c, padding='same').reshape(b, c, h, w).movedim(1, -1)
        a = f.conv2d(x.abs(), k.abs(), groups=b * c, padding='same').reshape(b, c, h, w).movedim(1, -1)
        n = f.conv2d(one, one, padding='same').movedim(1, -1)
    return s, a, n


def xcorr_interval(s, a, n, fmt, c=1.0):
    """[lo, hi] of the stored correlation: the kernel sums the n taps of an output one after the other with fmaf in
    fp32 (n roundings), so it lies within gamma_n * A, gamma_n = n u / (1 - n u), u = 2^-24, of S; then one rounding
    to the storage format (tf32 in tf32 mode, fp16 with its +-inf)."""
    an = a * (n / (1.0 - n * 2.0 ** -24))
    z = torch.zeros(s.shape[-1], dtype=torch.float32)
    return interval(s, an, z + 1.0, z, 1.0, fmt, c)


def xcorr_min_c(got, s, a, n, fmt, ladder=(0.0, 0.125, 0.25, 0.5, 1.0)):
    """Smallest c of the ladder (in units of gamma_n * A) for which every stored correlation passes (inf: none)."""
    got = got.to(s.device).float()
    for c in ladder:
        lo, hi = xcorr_interval(s, a, n, fmt, c)
        if not bool(violations(got, lo, hi).any()):
            return c
    return math.inf


# ------------------------------------------------------------------------------------------------ bilinear x2
def bilinear_coord(n):
    """The kernel's fp32 source coordinates (bilinear_coord in net.cu) of the 2n outputs of an extent n, align_corners
    True: f = fp32(fp32(n - 1) / fp32(2n - 1)) * o in fp32, i0 = min(int(f), n - 1), i1 = min(i0 + 1, n - 1),
    l1 = clamp(f - i0, 0, 1). PyTorch evaluates float32 up-sampling with the same expressions
    (area_pixel_compute_scale / guard_index_and_lambda). Returns (i0, i1) int64 tensors and l1 float32."""
    o = torch.arange(2 * n, dtype=torch.float32)
    s = torch.tensor(float(n - 1), dtype=torch.float32) / torch.tensor(float(2 * n - 1), dtype=torch.float32)
    f = s * o
    i0 = torch.clamp(f.to(torch.int64), max=n - 1)
    i1 = torch.clamp(i0 + 1, max=n - 1)
    l1 = torch.clamp(f - i0.to(torch.float32), 0.0, 1.0)
    return i0, i1, l1


def _lerp_matrix(n, device):
    """(2n, n) float64 matrix of the fp32 weights (1 - l1 in fp32, l1) at (i0, i1)."""
    i0, i1, l1 = bilinear_coord(n)
    m = torch.zeros((2 * n, n), dtype=torch.float64)
    r = torch.arange(2 * n)
    m[r, i0] += (1.0 - l1).double()
    m[r, i1] += l1.double()
    return m.to(device)


def bilinear_x2(x):
    """Bilinear x2 up-sampling with align_corners=True of a channels-last (N, H, W, C) tensor, in float64 with the
    kernel's (and PyTorch float32's) fp32 coordinates and weights, and the matching |.|-sum for the allowance (the
    weights are non-negative). F.interpolate on float64 would take float64 coordinates instead: at extent 64 they move
    a weight by up to about 2^-17, more than the fp32 evaluation's own error, so they are not what the kernel is
    held to. tests/test_layer_ref_host.py shows that this equals F.interpolate of float32 inputs."""
    n, h, w, c = x.shape
    mh, mw = _lerp_matrix(h, x.device), _lerp_matrix(w, x.device)
    xd = x.double()
    r = torch.einsum('yh,nhwc,xw->nyxc', mh, xd, mw)
    a = torch.einsum('yh,nhwc,xw->nyxc', mh, xd.abs(), mw)
    return r, a
