"""Host-side wrapper of the C-ABI network handle and of the HBM pipeline kernels.

PyTorch is used for device memory, streams and (in the multi-GPU driver) torch.distributed only; every kernel
that touches data is launched through ``libbiu_b200.so``. There is no CPU fallback.
"""
import ctypes
import warnings

import numpy as np
import torch

from . import _lib

KIND = {'unet2d': 0, 'siam2d': 1, 'unet3d': 2, 'mo3d': 3, 'unet2d_v0': 4, 'attunet2d': 5, 'mo2d': 6, 'nested2d': 7,
        'nested2d_3l': 8}
KIND_2D = ('unet2d', 'siam2d', 'unet2d_v0', 'attunet2d', 'mo2d', 'nested2d', 'nested2d_3l')
PRECISION = {'bf16': 0, 'tf32': 1, 'fp32': 2, 'fp16': 3}
SIAM_MODE = {'concat': 0, 'max': 1, 'control': 2, 'corr': 3}
ACT = {None: 0, 'none': 0, 'sigmoid': 1, 'tanh': 2, 'relu': 3}
HIST_BINS = 65536


def _require_cuda(device):
    device = torch.device(device)
    if device.type != 'cuda':
        raise RuntimeError(f"bio_image_unet_b200 runs on CUDA devices only (got '{device}'); there is no CPU fallback")
    if not torch.cuda.is_available():
        raise RuntimeError('bio_image_unet_b200: no CUDA device is available; there is no CPU fallback')
    return device


class Engine:
    """One network (weights folded + packed on the device) able to run batches of tiles.

    heads: list of (name, channels, activation) — a single ('', out_channels, 'sigmoid') entry for
    Unet / Siam_UNet / UNet3D, the ``output_heads`` dict entries for MultiOutputUnet3D.
    precision: 'bf16' | 'fp16' (tcgen05 operands and stored activations in that format, fp32 accumulation and
    BatchNorm / activation; fp16 keeps tf32's 10 mantissa bits, stores beyond +-65504 become +-inf) | 'tf32' (fp32
    storage) | 'fp32' (CUDA-core kernels).
    """

    def __init__(self, kind, state_dict, n_filter, in_channels=1, heads=(('', 1, 'sigmoid'),), siam_mode='concat',
                 use_interpolation=False, precision='bf16', device='cuda:0'):
        if precision not in PRECISION:
            raise ValueError(f"precision must be one of {list(PRECISION)} (got {precision!r})")
        self.device = _require_cuda(device)
        self.lib = _lib.load()
        if kind == 'siam2d' and siam_mode not in SIAM_MODE:
            raise NotImplementedError('Unknown mode: {}'.format(siam_mode))   # siam_unet/siam_unet.py:124
        self.kind, self.precision = kind, precision
        self.in_channels = int(in_channels)
        self.heads = [(str(n), int(c), a) for n, c, a in heads]
        self.head_total = sum(c for _, c, _ in self.heads)
        n_heads = len(self.heads)
        ch = (ctypes.c_int * n_heads)(*[c for _, c, _ in self.heads])
        ac = (ctypes.c_int * n_heads)(*[ACT[a] for _, _, a in self.heads])
        nm = (ctypes.c_char_p * n_heads)(*[n.encode() for n, _, _ in self.heads])
        with torch.cuda.device(self.device):
            self.handle = self.lib.biu_net_create(KIND[kind], int(n_filter), self.in_channels, n_heads, ch, ac, nm,
                                                  SIAM_MODE.get(siam_mode, 0), int(bool(use_interpolation)),
                                                  PRECISION[precision])
            if not self.handle:
                raise _lib.BiuError(_lib.last_error())
            for name, t in state_dict.items():
                if not torch.is_tensor(t) or not t.is_floating_point():
                    continue   # num_batches_tracked etc.
                a = np.ascontiguousarray(t.detach().to('cpu', torch.float32).numpy())
                shape = (ctypes.c_longlong * max(a.ndim, 1))(*(a.shape if a.ndim else (1,)))
                _lib.check(self.lib.biu_net_set_param(self.handle, name.encode(), a.ctypes.data_as(ctypes.c_void_p),
                                                      max(a.ndim, 1), shape), 'biu_net_set_param')
            _lib.check(self.lib.biu_net_finalize(self.handle), 'load_state_dict')
        self.batch = 0
        self.tile = None
        self.workspace = None
        self.fallback_ops = 0
        self._fallback_checked = False

    def plan(self, batch, tile, siam_shared=0):
        """tile: (h, w) or (d, h, w). siam_shared = tiles per frame: Siam_UNet in 'single' mode, the twin encoder runs
        once over the batch + siam_shared unique tiles of `batch` consecutive pairs (see biu_net_set_siam_shared)."""
        d, h, w = (1, *tile) if len(tile) == 2 else tile
        if self.kind == 'siam2d' or siam_shared:
            _lib.check(self.lib.biu_net_set_siam_shared(self.handle, int(siam_shared)), 'biu_net_set_siam_shared')
        self.siam_shared = int(siam_shared)
        with torch.cuda.device(self.device):
            nbytes = self.lib.biu_net_plan(self.handle, int(batch), int(d), int(h), int(w))
            if nbytes < 0:
                msg = _lib.last_error()
                if 'concatenation failed' in msg:
                    raise ValueError('concatenation failed: wrong dimensions')   # unet/unet.py:67
                raise _lib.BiuError(msg)
            if self.workspace is None or self.workspace.numel() < nbytes:
                self.workspace = None
                self.workspace = torch.zeros(int(nbytes), dtype=torch.uint8, device=self.device)
            else:
                self.workspace.zero_()
        self.batch, self.tile = int(batch), (int(d), int(h), int(w))
        self._fallback_checked = False
        return nbytes

    def forward(self, tiles, tiles_prev=None, want_val=False, want_u8=True):
        """tiles: (batch, in_channels, [d,] h, w) uint8 or float32 device tensor, exactly `batch` of the plan.
        Returns (val float32 | None, u8 | None), planar (batch, head_total, [d,] h, w)."""
        assert self.batch > 0, 'plan() first'
        assert tiles.is_cuda and tiles.is_contiguous()
        in_kind = 0 if tiles.dtype == torch.uint8 else 1
        if in_kind == 1 and tiles.dtype != torch.float32:
            raise TypeError('tiles must be uint8 or float32')
        d, h, w = self.tile
        n_in = self.batch + getattr(self, 'siam_shared', 0)
        assert tiles.numel() == n_in * self.in_channels * d * h * w, (tiles.shape, self.batch, self.tile)
        spatial = (h, w) if self.kind in KIND_2D else (d, h, w)
        shape = (self.batch, self.head_total, *spatial)
        val = torch.empty(shape, dtype=torch.float32, device=self.device) if want_val else None
        u8 = torch.empty(shape, dtype=torch.uint8, device=self.device) if want_u8 else None
        with torch.cuda.device(self.device):
            _lib.check(self.lib.biu_net_forward(self.handle, _lib.ptr(tiles), in_kind, _lib.ptr(tiles_prev),
                                                _lib.ptr(val), _lib.ptr(u8), _lib.ptr(self.workspace),
                                                _lib.stream_ptr()), 'biu_net_forward')
        if not self._fallback_checked:
            self._fallback_checked = True
            self.fallback_ops = int(self.lib.biu_net_fallback_ops(self.handle))
            if self.fallback_ops > 0 and self.precision != 'fp32':
                warnings.warn(f"bio_image_unet_b200: {self.fallback_ops} layer(s) of this {self.kind} network "
                              f"(n_filter / channel counts or tile shape outside what the tcgen05 kernels take) run on "
                              f"the roughly 10x slower CUDA-core kernels in precision='{self.precision}'; results are "
                              f"unaffected.", RuntimeWarning, stacklevel=3)
        return val, u8

    def debug_activation(self, name, channels, level, images=None):
        """Test hook: NHWC activation buffer `name` as a float32 host array (images, [d,] h, w, channels). images
        defaults to the batch; a twin-encoder buffer of Siam_UNet holds 2 * batch images ([current | previous]), or
        batch + siam_shared with the shared encoder."""
        images = self.batch if images is None else int(images)
        d, h, w = self.tile
        dd = max(d >> level, 1) if self.kind in ('unet3d', 'mo3d') else 1
        hh, ww = h >> level, w >> level
        esz = 2 if self.precision in ('bf16', 'fp16') else 4
        n = images * dd * hh * ww * channels
        host = np.empty(n * esz, dtype=np.uint8)
        torch.cuda.synchronize(self.device)
        _lib.check(self.lib.biu_net_debug_copy(self.handle, name.encode(), _lib.ptr(self.workspace),
                                               host.ctypes.data_as(ctypes.c_void_p), host.nbytes))
        if esz == 2:
            dt = torch.float16 if self.precision == 'fp16' else torch.bfloat16
            t = torch.from_numpy(host.view(np.int16).copy()).view(dt).float().numpy()
        else:
            t = host.view(np.float32)
        return t.reshape(images, dd, hh, ww, channels)

    def set_debug_stop(self, last_op):
        """Test hook: the following forwards return after op `last_op` of the layer program (-1: run all of it), so
        that what that op wrote can be read before a later op reuses the buffer. out_val / out_u8 are not written by
        a stopped forward, and read_profile() refuses it."""
        _lib.check(self.lib.biu_net_set_debug_stop(self.handle, int(last_op)), 'biu_net_set_debug_stop')

    def set_profile(self, on):
        """Bracket every op of the following forwards with CUDA events (read them with read_profile())."""
        _lib.check(self.lib.biu_net_set_profile(self.handle, int(on)))

    def read_profile(self, max_ops=128):
        """(kinds, ms) of the last profiled forward: op kind (+16: ran on the CUDA-core fallback, +32: fused into the
        previous kernel) and duration of every op of the layer program."""
        kinds = (ctypes.c_int * max_ops)()
        ms = (ctypes.c_float * max_ops)()
        n_ops = ctypes.c_int(0)
        _lib.check(self.lib.biu_net_profile_read(self.handle, max_ops, kinds, ms, ctypes.byref(n_ops)))
        return list(kinds[:n_ops.value]), list(ms[:n_ops.value])

    def set_force_direct(self, on):
        _lib.check(self.lib.biu_net_set_force_direct(self.handle, int(on)))

    def set_fuse_pool(self, on):
        _lib.check(self.lib.biu_net_set_fuse_pool(self.handle, int(on)))

    def close(self):
        if getattr(self, 'handle', None):
            self.lib.biu_net_destroy(self.handle)
            self.handle = None
        self.workspace = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ----------------------------------------------------------------------------------------------------------------
# HBM pipeline wrappers (all stream-ordered on torch's current stream)
# ----------------------------------------------------------------------------------------------------------------
_I32_CACHE = {}


def _dev_i32(values, device):
    """Device int32 array of tile starts. Cached: building it is a synchronous pageable H2D copy, which would stall
    the launching thread behind all queued work once per call (the starts repeat for every chunk of a movie)."""
    key = (tuple(int(v) for v in values), str(device))
    t = _I32_CACHE.get(key)
    if t is None:
        if len(_I32_CACHE) > 256:
            _I32_CACHE.clear()
        t = torch.tensor(list(key[0]), dtype=torch.int32, device=device)
        _I32_CACHE[key] = t
    return t


_I64_CACHE = {}


def _dev_i64(values, device):
    """Device int64 index tensor (frame selections of the Siam pairs), cached like _dev_i32."""
    key = (tuple(int(v) for v in values), str(device))
    t = _I64_CACHE.get(key)
    if t is None:
        if len(_I64_CACHE) > 64:
            _I64_CACHE.clear()
        t = torch.tensor(list(key[0]), dtype=torch.int64, device=device)
        _I64_CACHE[key] = t
    return t


def histogram(frames):
    """frames: (F, ...) uint8/uint16 device tensor -> (F, 65536) int32 counts."""
    lib = _lib.load()
    assert frames.is_cuda and frames.is_contiguous()
    if frames.dtype not in (torch.uint8, torch.uint16):
        raise TypeError(f'only uint8 / uint16 stacks are normalised on the device (got {frames.dtype})')
    f = frames.shape[0]
    hist = torch.empty((f, HIST_BINS), dtype=torch.int32, device=frames.device)
    with torch.cuda.device(frames.device):
        _lib.check(lib.biu_histogram(_lib.ptr(frames), frames.element_size(), frames[0].numel(), f, _lib.ptr(hist),
                                     _lib.stream_ptr()), 'biu_histogram')
    return hist


def hist_sum(hist):
    lib = _lib.load()
    out = torch.empty((1, HIST_BINS), dtype=torch.int32, device=hist.device)
    with torch.cuda.device(hist.device):
        _lib.check(lib.biu_hist_sum(_lib.ptr(hist), hist.shape[0], _lib.ptr(out), _lib.stream_ptr()), 'biu_hist_sum')
    return out


def norm_lut(hist_bounds, hist_range, frames, q_lo, q_hi, invert):
    """LUTs (frames, 65536) uint8 and params (frames, 4) float64 {lo, hi, mn, mx}. A histogram with a single row
    is shared by all frames."""
    lib = _lib.load()
    dev = hist_bounds.device
    lut = torch.empty((frames, HIST_BINS), dtype=torch.uint8, device=dev)
    params = torch.empty((frames, 4), dtype=torch.float64, device=dev)
    bs = HIST_BINS if hist_bounds.shape[0] > 1 else 0
    rs = HIST_BINS if hist_range.shape[0] > 1 else 0
    with torch.cuda.device(dev):
        _lib.check(lib.biu_norm_lut(_lib.ptr(hist_bounds), _lib.ptr(hist_range), bs, rs, frames, float(q_lo),
                                    float(q_hi), int(bool(invert)), _lib.ptr(lut), _lib.ptr(params),
                                    _lib.stream_ptr()), 'biu_norm_lut')
    return lut, params


def apply_lut(frames, lut):
    lib = _lib.load()
    out = torch.empty(frames.shape, dtype=torch.uint8, device=frames.device)
    stride = HIST_BINS if lut.shape[0] > 1 else 0
    with torch.cuda.device(frames.device):
        _lib.check(lib.biu_apply_lut(_lib.ptr(frames), frames.element_size(), frames[0].numel(), frames.shape[0],
                                     _lib.ptr(lut), stride, _lib.ptr(out), _lib.stream_ptr()), 'biu_apply_lut')
    return out


def gather_tiles(src, zs, ys, xs, tile, pad_mode):
    """src: (F, Z, H, W) uint8 device tensor; tile (pd, ph, pw); returns (F*nz*ny*nx, pd, ph, pw) uint8."""
    lib = _lib.load()
    f, z, h, w = src.shape
    pd, ph, pw = tile
    dev = src.device
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((f * len(zs) * len(ys) * len(xs), pd, ph, pw), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_gather_tiles(_lib.ptr(src), f, z, h, w, int(pad_mode), _lib.ptr(dzs), _lib.ptr(dys),
                                        _lib.ptr(dxs), len(zs), len(ys), len(xs), pd, ph, pw, _lib.ptr(out),
                                        _lib.stream_ptr()), 'biu_gather_tiles')
    return out


def gather_tiles_lut(raw, lut, zs, ys, xs, tile, pad_mode):
    """Normalisation fused into the tile gather: raw (F, Z, H, W) uint8 / uint16 device stack, lut (F | 1, 65536)
    uint8 tables of norm_lut(); returns the (F*nz*ny*nx, pd, ph, pw) uint8 tiles of the normalised stack without ever
    writing that stack."""
    lib = _lib.load()
    f, z, h, w = raw.shape
    pd, ph, pw = tile
    dev = raw.device
    assert raw.is_contiguous() and raw.dtype in (torch.uint8, torch.uint16)
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((f * len(zs) * len(ys) * len(xs), pd, ph, pw), dtype=torch.uint8, device=dev)
    stride = HIST_BINS if lut.shape[0] > 1 else 0
    with torch.cuda.device(dev):
        _lib.check(lib.biu_gather_tiles_lut(_lib.ptr(raw), raw.element_size(), _lib.ptr(lut), stride, f, z, h, w,
                                            int(pad_mode), _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs), len(zs), len(ys),
                                            len(xs), pd, ph, pw, _lib.ptr(out), _lib.stream_ptr()), 'biu_gather_tiles_lut')
    return out


def gather_tiles_tta(src, zs, ys, xs, tile, pad_mode, dims, t, lut=None):
    """gather_tiles (src uint8, lut None) or gather_tiles_lut (raw uint8 / uint16 stack and its tables) producing the
    tiles under test-time augmentation transform t (2D, dims 2: bit 0 flips x, 1 flips y, 2 transposes; 3D: bits 0-2
    flip x, y, z). t = 0 gives the plain tiles."""
    lib = _lib.load()
    f, z, h, w = src.shape
    pd, ph, pw = tile
    dev = src.device
    assert src.is_contiguous() and src.dtype in (torch.uint8, torch.uint16)
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((f * len(zs) * len(ys) * len(xs), pd, ph, pw), dtype=torch.uint8, device=dev)
    stride = 0 if lut is None or lut.shape[0] == 1 else HIST_BINS
    with torch.cuda.device(dev):
        _lib.check(lib.biu_gather_tiles_tta(_lib.ptr(src), src.element_size(), _lib.ptr(lut), stride, f, z, h, w,
                                            int(pad_mode), _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs), len(zs), len(ys),
                                            len(xs), pd, ph, pw, int(dims), int(t), _lib.ptr(out), _lib.stream_ptr()),
                   'biu_gather_tiles_tta')
    return out


def gather_tiles_f32_tta(src, zs, ys, xs, tile, dims, t):
    """gather_tiles_f32 producing the patches under transform t (see gather_tiles_tta)."""
    lib = _lib.load()
    f, z, h, w = src.shape
    pd, ph, pw = tile
    dev = src.device
    assert src.is_contiguous() and src.dtype == torch.float32
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((f * len(zs) * len(ys) * len(xs), pd, ph, pw), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_gather_tiles_f32_tta(_lib.ptr(src), f, z, h, w, _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs),
                                                len(zs), len(ys), len(xs), pd, ph, pw, int(dims), int(t), _lib.ptr(out),
                                                _lib.stream_ptr()), 'biu_gather_tiles_f32_tta')
    return out


def tta_accumulate(val, acc, dims, t, p, passes, out_u8=None, out_f32=None):
    """Pass p of `passes` of the test-time augmentation merge. val: (n, C, [d,] h, w) float32 output of the net on
    the tiles of transform t; acc: fp32 buffer of val's shape (the running sum of T^-1(val) in pass order; written by
    pass 0, not needed when passes == 1). The last pass writes the mean to out_f32 and / or trunc(mean * 255) to
    out_u8 (tensors of val's shape)."""
    lib = _lib.load()
    assert val.is_contiguous() and val.dtype == torch.float32
    for o in (acc, out_u8, out_f32):
        assert o is None or (o.is_contiguous() and o.shape == val.shape)
    pd = val.shape[2] if val.dim() == 5 else 1
    with torch.cuda.device(val.device):
        _lib.check(lib.biu_tta_accumulate(_lib.ptr(val), val.shape[0] * val.shape[1], pd, val.shape[-2], val.shape[-1],
                                          int(dims), int(t), int(p), int(passes), _lib.ptr(acc), _lib.ptr(out_u8),
                                          _lib.ptr(out_f32), _lib.stream_ptr()), 'biu_tta_accumulate')


def stitch_mean_u8(tiles, frames, channels, out_hw, ys, xs, tile_hw):
    """tiles (F*ny*nx, C, ph, pw) uint8 -> (F, C, H, W) uint8, sum // count over covering tiles."""
    lib = _lib.load()
    dev = tiles.device
    dys, dxs = _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((frames, channels, out_hw[0], out_hw[1]), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_stitch_mean_u8(_lib.ptr(tiles), frames, channels, out_hw[0], out_hw[1], _lib.ptr(dys),
                                          _lib.ptr(dxs), len(ys), len(xs), tile_hw[0], tile_hw[1], _lib.ptr(out),
                                          _lib.stream_ptr()), 'biu_stitch_mean_u8')
    return out


def stitch_mod3_u8(tiles, out_zhw, zs, ys, xs, tile):
    lib = _lib.load()
    dev = tiles.device
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty(tuple(out_zhw), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_stitch_mod3_u8(_lib.ptr(tiles), out_zhw[0], out_zhw[1], out_zhw[2], _lib.ptr(dzs),
                                          _lib.ptr(dys), _lib.ptr(dxs), len(zs), len(ys), len(xs), tile[0], tile[1],
                                          tile[2], _lib.ptr(out), _lib.stream_ptr()), 'biu_stitch_mod3_u8')
    return out


def stitch_weighted_u8(tiles, frames, channels, out_zhw, zs, ys, xs, tile, w_d, w_h, w_w):
    """Engine-only weighted stitch: tiles (F*nz*ny*nx, C, pd, ph, pw) uint8 -> (F, C, Z, H, W) uint8,
    out = (sum w * v) // (sum w) over the covering tiles, w = w_d[tz] * w_h[ty] * w_w[tx], in exact integer arithmetic
    (0 where nothing covers an element). Starts may be negative; w_d / w_h / w_w have pd / ph / pw entries in [0, 1024]."""
    lib = _lib.load()
    dev = tiles.device
    pd, ph, pw = (int(v) for v in tile)
    tables = []
    for name, tab, n in (('w_d', w_d, pd), ('w_h', w_h, ph), ('w_w', w_w, pw)):
        tab = [int(v) for v in tab]
        if len(tab) != n:
            raise ValueError(f'{name} has {len(tab)} entries for a tile axis of {n}')
        if min(tab) < 0 or max(tab) > 1024:
            raise ValueError(f'{name} entries must lie in [0, 1024]')
        tables.append(_dev_i32(tab, dev))
    assert tiles.is_contiguous() and tiles.dtype == torch.uint8
    assert tiles.numel() == frames * len(zs) * len(ys) * len(xs) * channels * pd * ph * pw, (tiles.shape, tile)
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((frames, channels, *out_zhw), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_stitch_weighted_u8(_lib.ptr(tiles), frames, channels, out_zhw[0], out_zhw[1], out_zhw[2],
                                              _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs), len(zs), len(ys), len(xs),
                                              pd, ph, pw, *(_lib.ptr(t) for t in tables), _lib.ptr(out),
                                              _lib.stream_ptr()), 'biu_stitch_weighted_u8')
    return out


def stitch_ramp_f32(tiles, vols, channels, out_zhw, zs, ys, xs, tile, margin=16):
    lib = _lib.load()
    dev = tiles.device
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((vols, channels, *out_zhw), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_stitch_ramp_f32(_lib.ptr(tiles), vols, channels, out_zhw[0], out_zhw[1], out_zhw[2],
                                           _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs), len(zs), len(ys), len(xs),
                                           tile[0], tile[1], tile[2], int(margin), _lib.ptr(out), _lib.stream_ptr()),
                   'biu_stitch_ramp_f32')
    return out


def norm_lut_f32(hist_bounds, hist_range, frames, q_lo, q_hi, mode):
    """float32 LUTs (frames, 65536) of multi_output_unet3d's normalisation; mode 0 'single', 1 'first'/'all'."""
    lib = _lib.load()
    dev = hist_bounds.device
    lut = torch.empty((frames, HIST_BINS), dtype=torch.float32, device=dev)
    params = torch.empty((frames, 4), dtype=torch.float64, device=dev)
    bs = HIST_BINS if hist_bounds.shape[0] > 1 else 0
    rs = HIST_BINS if hist_range.shape[0] > 1 else 0
    with torch.cuda.device(dev):
        _lib.check(lib.biu_norm_lut_f32(_lib.ptr(hist_bounds), _lib.ptr(hist_range), bs, rs, frames, float(q_lo),
                                        float(q_hi), int(mode), _lib.ptr(lut), _lib.ptr(params), _lib.stream_ptr()),
                   'biu_norm_lut_f32')
    return lut, params


def apply_lut_f32(frames, lut):
    lib = _lib.load()
    out = torch.empty(frames.shape, dtype=torch.float32, device=frames.device)
    stride = HIST_BINS if lut.shape[0] > 1 else 0
    with torch.cuda.device(frames.device):
        _lib.check(lib.biu_apply_lut_f32(_lib.ptr(frames), frames.element_size(), frames[0].numel(), frames.shape[0],
                                         _lib.ptr(lut), stride, _lib.ptr(out), _lib.stream_ptr()), 'biu_apply_lut_f32')
    return out


def gather_tiles_f32(src, zs, ys, xs, tile):
    """src (F, Z, H, W) float32 -> (F*nz*ny*nx, pd, ph, pw) float32 (patches lie inside the volume)."""
    lib = _lib.load()
    f, z, h, w = src.shape
    pd, ph, pw = tile
    dev = src.device
    dzs, dys, dxs = _dev_i32(zs, dev), _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((f * len(zs) * len(ys) * len(xs), pd, ph, pw), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_gather_tiles_f32(_lib.ptr(src), f, z, h, w, _lib.ptr(dzs), _lib.ptr(dys), _lib.ptr(dxs),
                                            len(zs), len(ys), len(xs), pd, ph, pw, _lib.ptr(out), _lib.stream_ptr()),
                   'biu_gather_tiles_f32')
    return out


def stitch_margin_f32(tiles, src_index, frames, channels, out_hw, ys, xs, tile_hw, fill, margin=20):
    """multi_output_unet/predict.py:230-285. tiles (P, C, ph, pw) float32; src_index (frames, ny, nx) int32 device
    tensor of flat patch indices; fill: 1-element float32 device tensor. Returns (frames, C, H, W) float32."""
    lib = _lib.load()
    dev = tiles.device
    dys, dxs = _dev_i32(ys, dev), _dev_i32(xs, dev)
    out = torch.empty((frames, channels, out_hw[0], out_hw[1]), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(lib.biu_stitch_margin_f32(_lib.ptr(tiles), _lib.ptr(src_index), frames, channels, out_hw[0], out_hw[1],
                                             _lib.ptr(dys), _lib.ptr(dxs), len(ys), len(xs), tile_hw[0], tile_hw[1],
                                             int(margin), _lib.ptr(fill), _lib.ptr(out), _lib.stream_ptr()),
                   'biu_stitch_margin_f32')
    return out


def normalize_f32(frames, mode, q_lo, q_hi, invert, want_f32=False):
    """Percentile normalisation of a float32 (F, ...) device stack to uint8 (unet/predict.py:122-150 as numpy
    evaluates it on float32 data). mode: 'single' | 'first' | 'all'. Returns (u8, float32 values | None, params)."""
    lib = _lib.load()
    assert frames.is_cuda and frames.is_contiguous() and frames.dtype == torch.float32
    f = frames.shape[0]
    n = frames[0].numel()
    dev = frames.device
    m = {'single': 0, 'first': 1, 'all': 2}[mode]
    scratch = torch.empty(int(lib.biu_normalize_f32_scratch_bytes(n, f)), dtype=torch.uint8, device=dev)
    params = torch.empty((f if m == 0 else 1, 4), dtype=torch.float32, device=dev)
    out_u8 = torch.empty(frames.shape, dtype=torch.uint8, device=dev)
    out_f32 = torch.empty(frames.shape, dtype=torch.float32, device=dev) if want_f32 else None
    with torch.cuda.device(dev):
        _lib.check(lib.biu_normalize_f32(_lib.ptr(frames), n, f, m, float(q_lo), float(q_hi), int(bool(invert)),
                                         _lib.ptr(scratch), _lib.ptr(params), _lib.ptr(out_u8), _lib.ptr(out_f32),
                                         _lib.stream_ptr()), 'biu_normalize_f32')
    return out_u8, out_f32, params
