"""Device pipeline shared by the 2D predictors: normalise -> split -> batched forward -> stitch.

Reference: unet/predict.py:115-229 (and the per-pair variant siam_unet/predict.py:125-240). All heavy steps run
as CUDA kernels through the C-ABI; this module only sequences them and does the (tiny) index arithmetic.
"""
import functools

import numpy as np
import torch

from . import engine as E
from . import tiling


def to_device_stack(frames_np, device):
    """(F, H, W) uint8 / uint16 / float32 host array (numpy, or a torch tensor - ideally pinned) -> device tensor."""
    if torch.is_tensor(frames_np):
        if frames_np.dtype not in (torch.uint8, torch.uint16, torch.float32):
            raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 / float32 stacks on the device; got {frames_np.dtype}')
        return frames_np.contiguous().to(device, non_blocking=True)
    if frames_np.dtype not in (np.uint8, np.uint16, np.float32):
        raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 / float32 stacks on the device; got '
                        f'{frames_np.dtype}. Convert the stack (e.g. to uint16 or float32) before calling Predict.')
    host = torch.from_numpy(np.ascontiguousarray(frames_np))
    try:
        host = host.pin_memory()
    except RuntimeError:
        pass
    return host.to(device, non_blocking=True)


class PinnedPool:
    """Reusable pinned host buffers, one per key, grown on demand. A view stays valid until the next call that uses
    the same key."""

    def __init__(self):
        self.bufs = {}

    def view(self, key, shape, dtype):
        """Pinned host tensor of the given shape and dtype."""
        n = int(np.prod(shape)) * dtype.itemsize
        buf = self.bufs.get(key)
        if buf is None or buf.numel() < n:
            buf = self.bufs[key] = torch.empty(n, dtype=torch.uint8, pin_memory=True)
        return buf[:n].view(dtype).view(*shape)

    def fetch(self, key, t):
        """Device tensor `t` copied to the host: a numpy view of the pinned buffer of `key`."""
        host = self.view(key, t.shape, t.dtype)
        host.copy_(t, non_blocking=True)
        torch.cuda.current_stream(t.device).synchronize()
        return host.numpy()

    def close(self):
        self.bufs = {}


TTA_MODES = (None, 'flips', 'dihedral')


def tta_codes(tta, dims, tile):
    """Transform codes of a predictor's `tta` setting, checked before any device work: None (no augmentation),
    'flips' (2D: the 4 flips of y and x, t = 0..3; 3D: the 8 flips of z, y and x, t = 0..7) or 'dihedral' (2D square
    tiles: all 8 symmetries of the square, t = 0..7; bit 2 transposes after the flips)."""
    if tta is None:
        return None
    if not isinstance(tta, str) or tta not in TTA_MODES:
        raise ValueError(f"tta must be one of {list(TTA_MODES)} (got {tta!r})")
    if tta == 'flips':
        return list(range(4 if dims == 2 else 8))
    if dims != 2:
        raise ValueError("tta='dihedral' needs 2D tiles: the 3D predictors take tta='flips' or None")
    if int(tile[-1]) != int(tile[-2]):
        raise ValueError(f"tta='dihedral' transposes tiles and needs square ones (got {tuple(tile)})")
    return list(range(8))


BLEND_MODES = (None, 'gaussian')


def blend_mode(blend):
    """A predictor's `blend` setting, checked before any device work: None (the reference's stitch) or 'gaussian'
    (overlapping tiles weighted by blend_tables, exact integer weighted mean of the uint8 result tiles)."""
    if blend is None:
        return None
    if not isinstance(blend, str) or blend not in BLEND_MODES:
        raise ValueError(f"blend must be one of {list(BLEND_MODES)} (got {blend!r})")
    return blend


@functools.lru_cache(maxsize=None)
def _gaussian_table(n):
    return tuple(int(v) for v in tiling.gaussian_weights(n))


def blend_tables(tile):
    """Per-axis weight tables (w_d, w_h, w_w) of blend='gaussian' for a 2D (th, tw) tile (w_d = [1]) or a 3D
    (pd, ph, pw) patch."""
    tile = tuple(int(v) for v in tile)
    return ((1,) if len(tile) == 2 else _gaussian_table(tile[0])), _gaussian_table(tile[-2]), _gaussian_table(tile[-1])


def stitch_2d(res_u8, frames, channels, out_hw, xs, ys, tile_hw, blend=None):
    """Stitch of the (frames * N, C, th, tw) uint8 result tiles of a 2D grid (xs: starts along rows, ys: along
    columns) into (frames, C, H, W): the reference's mean (blend None) or the weighted stitch of blend='gaussian'.
    One tile per frame (Siam_UNet on whole frames) has nothing to blend: both give the tile itself."""
    if blend is None or len(xs) * len(ys) == 1:
        return E.stitch_mean_u8(res_u8, frames, channels, out_hw, xs, ys, tile_hw)
    out = E.stitch_weighted_u8(res_u8, frames, channels, (1, *out_hw), [0], xs, ys, (1, *tile_hw),
                               *blend_tables(tile_hw))
    return out.view(frames, channels, *out_hw)


def tta_extra_bytes(tta, channels, tile, in_bytes=1):
    """Device bytes per tile that test-time augmentation adds to a batch: the float output of the forward, the fp32
    running sum and the transformed input tile."""
    if tta is None:
        return 0
    px = int(np.prod(tile))
    return 8 * int(channels) * px + int(in_bytes) * px


def _joined(outs):
    return None if not outs else outs[0] if len(outs) == 1 else torch.cat(outs)


def run_tiles(eng, tiles, tile_batch, prev_tiles=None, n_per=0, want_val=False, want_u8=True, on_val=None,
              progress=None):
    """Forward all tiles in batches of the planned `tile_batch` results (the tail batch is zero-padded) and return
    the (uint8, float) outputs of the head, trimmed to the tiles; an output that is not wanted is None. With `on_val`
    every batch's float output goes to on_val(start, val) instead: no uint8 output is made and both returned are None.

    prev_tiles: the second input of a two-input Siam_UNet, sliced like `tiles`. n_per: Siam_UNet with the shared twin
    encoder, n_per tiles per frame - tiles = [tiles of the previous frame of the first pair | tiles of the current
    frames], pair j = (tile j, tile j + n_per), so len(tiles) - n_per results, and the batch starting at pair s takes
    the unique tiles tiles[s : s + cnt + n_per]. progress: wraps the iterator over the batch starts."""
    if on_val is not None:
        want_val, want_u8 = True, False
    n = tiles.shape[0] - n_per
    starts = range(0, n, tile_batch)
    outs_u8, outs_val = [], []
    for s in (starts if progress is None else progress(starts)):
        cnt = min(tile_batch, n - s)
        t = tiles[s:s + cnt + n_per]
        p = None if prev_tiles is None else prev_tiles[s:s + cnt]
        if cnt < tile_batch:
            pad = torch.zeros((tile_batch - cnt, *t.shape[1:]), dtype=t.dtype, device=t.device)
            t = torch.cat((t, pad))
            p = None if p is None else torch.cat((p, pad))
        val, u8 = eng.forward(t.contiguous(), None if p is None else p.contiguous(), want_val=want_val, want_u8=want_u8)
        if on_val is not None:
            on_val(s, val[:cnt])
            continue
        if want_u8:
            outs_u8.append(u8[:cnt])
        if want_val:
            outs_val.append(val[:cnt])
    return _joined(outs_u8), _joined(outs_val)


def even_batch(total_tiles, budget_batch):
    """Tile batch for a job of `total_tiles`: as few forwards as the workspace budget allows, all of (almost) the same
    size - 288 tiles with room for 160 run as 2 x 144, not 160 + 128 padded to 160."""
    total_tiles, budget_batch = max(1, int(total_tiles)), max(1, int(budget_batch))
    n_fwd = -(-total_tiles // budget_batch)
    return -(-total_tiles // n_fwd)


class BatchPlanner:
    """Plan policy shared by the Session classes: the plan grows on demand, shrinks only when a job is at most half
    the planned batch (padding a 25-tile image to a 200-tile batch would cost 8x), and is never re-made for the
    shorter tail chunk of a movie (run_tiles pads that one)."""

    def __init__(self, engine, workspace_bytes, extra_per_tile=None):
        self.engine, self.workspace_bytes = engine, workspace_bytes
        self.tile, self.budget_batch, self.tile_batch = None, None, None
        self.plan_kwargs = {}                      # e.g. siam_shared=tiles per frame (Engine.plan)
        self.extra_per_tile = extra_per_tile       # tile -> bytes per tile outside the workspace (test-time augmentation)

    def budget(self, tile):
        """Largest tile batch the workspace budget holds for this tile size."""
        tile = tuple(int(v) for v in tile)
        key = (tile, tuple(sorted(self.plan_kwargs.items())))
        if self.tile != key:
            per_tile = self.engine.plan(1, tile) + (self.extra_per_tile(tile) if self.extra_per_tile else 0)
            self.budget_batch = int(max(1, self.workspace_bytes // max(per_tile, 1)))
            self.tile, self.tile_batch = key, None
        return self.budget_batch

    def ensure(self, tile, total_tiles):
        tile = tuple(int(v) for v in tile)
        self.budget(tile)
        target = even_batch(total_tiles, self.budget_batch)
        if self.tile_batch is None or target > self.tile_batch or 2 * target <= self.tile_batch:
            self.engine.plan(target, tile, **self.plan_kwargs)
            self.tile_batch = target
        return self.tile_batch


def predict_tiles(gather, run, n, codes, dims, out_dtype=torch.uint8):
    """Result tiles of one chunk of `n` tiles and the chunk's plain input tiles: (result, gather(0)). gather(t) makes
    the input tiles under transform t (t = 0: the plain tiles); run(tiles, on_val) is run_tiles on them, returning
    its (uint8, float) outputs.

    codes None: the plain tiles run once, and the result is the head's own output - its uint8, or its float output
    for out_dtype float32. Otherwise test-time augmentation: for every transform code t of `codes`, in ascending
    order, the same forwards as a plain prediction run on gather(t), and every batch's float output goes through
    T_t^-1 into one fp32 running sum of the chunk. The last pass writes the mean as uint8 (trunc(mean * 255), as the
    head does) or as float32 (out_dtype). Plans, tile batches and stitches are those of a plain prediction; the cost
    is len(codes) forwards per tile."""
    if codes is None:
        plain = gather(0)
        u8, val = run(plain, None)
        return (u8 if out_dtype == torch.uint8 else val), plain
    k = len(codes)
    bufs = {}
    for p, t in enumerate(codes):
        def on_val(s, val, p=p, t=t):
            if not bufs:
                shape = (n, *val.shape[1:])
                bufs['out'] = torch.empty(shape, dtype=out_dtype, device=val.device)
                bufs['acc'] = torch.empty(shape, dtype=torch.float32, device=val.device) if k > 1 else None
            cnt = val.shape[0]
            acc = None if bufs['acc'] is None else bufs['acc'][s:s + cnt]
            out = bufs['out'][s:s + cnt]
            E.tta_accumulate(val, acc, dims, t, p, k, out_u8=out if out_dtype == torch.uint8 else None,
                             out_f32=out if out_dtype == torch.float32 else None)
        tiles = gather(t)
        if t == 0:
            plain = tiles
        run(tiles, on_val)
    return bufs['out'], plain


def pick_tile_batch(eng, tile, total_tiles, budget_bytes):
    per_tile = eng.plan(1, tile)
    batch = int(max(1, min(total_tiles, budget_bytes // max(per_tile, 1))))
    eng.plan(batch, tile)
    return batch


def check_starts(starts, tile, extent):
    """The reference wraps negative uint16 starts when an undersized image is split into more than one tile and
    then fails on the slice assignment; report that as the same ValueError class up front."""
    for s in starts:
        if int(s) + tile > max(extent, tile):
            raise ValueError(f'could not broadcast tile: start {int(s)} + tile {tile} exceeds extent {extent} '
                             f'(image smaller than resize_dim with add_tile > 0)')


def predict_frames_2d(eng, frames, resize_dim, add_tile, out_channels, tile_batch, lut=None, pad_mode=0, tta=None,
                      blend=None):
    """frames: (F, H, W) contiguous device stack, already normalised to uint8 - or, with `lut` (its normalisation
    tables), the raw uint8 / uint16 stack: the normalisation is then fused into the tile gather and the normalised
    stack is never written. tta: transform codes of test-time augmentation (tta_codes) or None; blend: blend_mode()
    value. Returns ((F, C, H, W) uint8 device tensor, grid, tiles, result_tiles); `tiles` are the plain (t = 0)
    (F*N, 1, th, tw) tiles."""
    f, h, w = frames.shape
    th, tw = resize_dim
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, resize_dim, add_tile)
    check_starts(xs, th, h)
    check_starts(ys, tw, w)
    src = frames.view(f, 1, h, w)
    res_u8, tiles = predict_tiles(lambda t: E.gather_tiles_tta(src, [0], xs, ys, (1, th, tw), pad_mode, 2, t, lut=lut),
                                  lambda tl, on_val: run_tiles(eng, tl, tile_batch, on_val=on_val),
                                  f * n_x * n_y, tta, 2)
    out = stitch_2d(res_u8, f, out_channels, (h, w), xs, ys, (th, tw), blend)
    return out, (n_x, n_y, xs, ys), tiles, res_u8
