"""Host-side tile-grid arithmetic. Kept in numpy with the reference's exact expressions so that tile counts and
start indices are bit-identical (uint16 truncation of np.linspace included)."""
import numpy as np


def linspace_starts(extent, tile, count):
    """np.linspace(0, extent - tile, count).astype('uint16') — unet/predict.py:171-172."""
    return np.linspace(0, extent - tile, count).astype('uint16')


def grid_2d(height, width, resize_dim, add_tile):
    """(N_x, N_y, X_start, Y_start) of unet/predict.py:154-155,171-172 and siam_unet/predict.py:92-95,183-184.
    Note the reference's naming: 'x' runs along image rows (axis 1 of the stack), 'y' along columns."""
    n_x = int(np.ceil(height / resize_dim[0])) + add_tile
    n_y = int(np.ceil(width / resize_dim[1])) + add_tile
    return n_x, n_y, linspace_starts(height, resize_dim[0], n_x), linspace_starts(width, resize_dim[1], n_y)


def grid_3d(vol_shape, resize_dim, add_patch):
    """(N_z, N_x, N_y, Z_start, X_start, Y_start) of unet3d/predict.py:121-126,140-142 — including the
    as-written quirk that N_x is incremented when N_z > 1 and again when N_x > 1."""
    n_z = int(np.ceil(vol_shape[0] / resize_dim[0])) + add_patch
    n_x = int(np.ceil(vol_shape[1] / resize_dim[1])) + add_patch
    n_y = int(np.ceil(vol_shape[2] / resize_dim[2])) + add_patch
    if n_z > 1:
        n_x += add_patch
    if n_x > 1:
        n_x += add_patch
    if n_y > 1:
        n_y += add_patch
    return (n_z, n_x, n_y, linspace_starts(vol_shape[0], resize_dim[0], n_z),
            linspace_starts(vol_shape[1], resize_dim[1], n_x), linspace_starts(vol_shape[2], resize_dim[2], n_y))


def strided_starts(extent, patch, overlap_factor):
    """Patch starts along one axis of multi_output_unet3d/predict.py:134-147: uniform stride
    int(patch * (1 - overlap)), plus a final start flush with the far edge when the tail is uncovered."""
    stride = max(1, int(patch * (1 - overlap_factor)))
    starts = list(range(0, max(extent - patch + 1, 1), stride))
    if starts[-1] + patch < extent:
        starts.append(extent - patch)
    return starts


def gaussian_weights(n):
    """Centre-weighted blend table of a tile axis of length n >= 1 (engine-only `blend='gaussian'`), in float64:
    sigma = n / 8, g(i) = 1024 * exp(-(i - (n - 1) / 2)^2 / (2 sigma^2)), w(i) = max(1, floor(g(i) + 0.5)) as int32.
    Symmetric (w(i) = w(n - 1 - i)), every value in [1, 1024]; n = 1 gives [1024]."""
    n = int(n)
    if n < 1:
        raise ValueError(f'a tile axis has at least one element (got {n})')
    i = np.arange(n, dtype=np.float64)
    sigma = n / 8
    g = 1024.0 * np.exp(-(i - (n - 1) / 2) ** 2 / (2 * sigma ** 2))
    return np.maximum(1, np.floor(g + 0.5)).astype(np.int32)


def shard_range(n_items, rank, world_size):
    """Contiguous, balanced [start, stop) slice of n_items for `rank` (frames / z-rows of patches / volumes)."""
    base, rem = divmod(n_items, world_size)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def zslab_plan(z_starts, patch_d, vol_z, world_size):
    """Sharding of the z-rows of a 3D patch grid (the outermost loop of unet3d/predict.py:146,180) over ranks.

    Returns one dict per rank: rows (lo, hi) = its z-rows; slab (a, b) = the input planes those rows touch; own
    (lo, hi) = the output planes it stitches (the planes of its slab that no lower rank covers: the `own` ranges
    partition [0, vol_z)); borrow = {higher rank: [z-rows]} whose patches reach down into `own` and must be received
    before stitching. Rows never need to travel upwards: a rank's `own` starts where the previous rank's last row
    ends."""
    zs = [int(v) for v in z_starts]
    n_z = len(zs)
    rows = [shard_range(n_z, r, world_size) for r in range(world_size)]

    def row_end(zi):
        return min(vol_z, zs[zi] + patch_d)

    plans = []
    for lo, hi in rows:
        if hi <= lo:
            plans.append(dict(rows=(lo, hi), slab=(0, 0), own=(0, 0), borrow={}))
            continue
        a, b = zs[lo], row_end(hi - 1)
        own_lo = min(max(a, row_end(lo - 1)) if lo > 0 else 0, b)
        plans.append(dict(rows=(lo, hi), slab=(a, b), own=(own_lo, b), borrow={}))
    for r, p in enumerate(plans):
        if p['own'][1] <= p['own'][0]:
            continue
        for s in range(r + 1, world_size):
            need = [zi for zi in range(*rows[s]) if zs[zi] < p['own'][1]]
            if need:
                p['borrow'][s] = need
    return plans
