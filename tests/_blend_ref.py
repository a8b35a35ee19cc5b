"""numpy reference of the engine-only weighted overlap stitch (blend='gaussian'; not part of the reference package, so
not in oracle/): out = (sum w * v) // (sum w) over the tiles covering an element, w = w_d[tz] * w_h[ty] * w_w[tx],
exact unsigned 64-bit integers, 0 where nothing covers an element or the weights sum to 0."""
import math

import numpy as np


def gaussian_table(n):
    """The blend table of a tile axis of length n, evaluated element by element with the math module."""
    sigma = n / 8
    c = (n - 1) / 2
    return np.array([max(1, math.floor(1024.0 * math.exp(-(i - c) ** 2 / (2 * sigma ** 2)) + 0.5)) for i in range(n)],
                    dtype=np.int64)


def stitch_weighted(tiles, frames, channels, out_zhw, zs, ys, xs, tile, w_d, w_h, w_w):
    """tiles (frames * nz * ny * nx, C, pd, ph, pw) uint8 (any shape of that size) -> (frames, C, Z, H, W) uint8.
    Starts may be negative and tiles may reach past the output."""
    pd, ph, pw = tile
    z, h, w = out_zhw
    tiles = np.asarray(tiles).reshape(frames, len(zs) * len(ys) * len(xs), channels, pd, ph, pw)
    wt = (np.asarray(w_d, np.uint64)[:, None, None] * np.asarray(w_h, np.uint64)[None, :, None] *
          np.asarray(w_w, np.uint64)[None, None, :])
    num = np.zeros((frames, channels, z, h, w), np.uint64)
    den = np.zeros((z, h, w), np.uint64)
    n = 0
    for z0 in (int(v) for v in zs):
        for y0 in (int(v) for v in ys):
            for x0 in (int(v) for v in xs):
                a0, a1 = max(z0, 0), min(z0 + pd, z)
                b0, b1 = max(y0, 0), min(y0 + ph, h)
                c0, c1 = max(x0, 0), min(x0 + pw, w)
                if a1 > a0 and b1 > b0 and c1 > c0:
                    ws = wt[a0 - z0:a1 - z0, b0 - y0:b1 - y0, c0 - x0:c1 - x0]
                    v = tiles[:, n, :, a0 - z0:a1 - z0, b0 - y0:b1 - y0, c0 - x0:c1 - x0].astype(np.uint64)
                    num[:, :, a0:a1, b0:b1, c0:c1] += ws * v
                    den[a0:a1, b0:b1, c0:c1] += ws
                n += 1
    out = np.where(den > 0, num // np.maximum(den, 1), 0)
    return out.astype(np.uint8)


def stitch_weighted_2d(tiles, frames, out_hw, xs, ys, tile_hw, w_h, w_w):
    """2D form: tiles (frames * n_x * n_y, C, th, tw); xs starts along rows, ys along columns (the grid_2d naming).
    Returns (frames, C, H, W)."""
    tiles = np.asarray(tiles)
    c = tiles.shape[1]
    out = stitch_weighted(tiles, frames, c, (1, *out_hw), [0], xs, ys, (1, *tile_hw), [1], w_h, w_w)
    return out[:, :, 0]
