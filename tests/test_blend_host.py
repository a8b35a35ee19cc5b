"""Gaussian overlap blending without a GPU: the weight tables, the numpy weighted stitch (unit tables reduce it to the
reference's mean stitch, the tile-edge step it removes), its locality under the 3D z-slab plan, and the `blend`
argument checks of every predictor."""
import numpy as np
import pytest

from bio_image_unet_b200 import pipeline2d as P
from bio_image_unet_b200 import tiling
from oracle import pipeline as opipe
from tests import _blend_ref as B
from tests.test_host_logic import _random_zslab_cases

# the 2D grids of test_gpu_unet.test_stitch_mean_bit_exact: add_tile 0..14, undersized images, starts that are not
# multiples of 16, more than eight tiles over one 16-pixel run
GRIDS_2D = [(70, 90, 32, 48, 1, 1), (64, 64, 32, 32, 2, 2), (20, 100, 32, 48, 0, 1), (33, 47, 16, 16, 3, 1),
            (96, 200, 32, 160, 14, 1), (64, 256, 32, 64, 1, 2)]


def test_gaussian_tables():
    for n in range(1, 1025):
        w = tiling.gaussian_weights(n)
        assert w.dtype == np.int32 and w.shape == (n,)
        assert np.array_equal(w, B.gaussian_table(n)), n
        assert np.array_equal(w, w[::-1]), n
        assert w.min() >= 1 and w.max() <= 1024, n
    assert list(tiling.gaussian_weights(1)) == [1024]
    assert list(tiling.gaussian_weights(8)) == [2, 45, 332, 904, 904, 332, 45, 2]
    with pytest.raises(ValueError):
        tiling.gaussian_weights(0)


def test_blend_tables():
    assert P.blend_tables((32, 48)) == ((1,), tuple(tiling.gaussian_weights(32)), tuple(tiling.gaussian_weights(48)))
    wd, wh, ww = P.blend_tables((8, 16, 24))
    assert (wd, wh, ww) == tuple(tuple(int(v) for v in tiling.gaussian_weights(n)) for n in (8, 16, 24))


@pytest.mark.parametrize('h,w,th,tw,add,c', GRIDS_2D)
def test_unit_tables_equal_mean_stitch(h, w, th, tw, add, c):
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
    f = 2
    tiles = np.random.default_rng(h * w + add).integers(0, 256, (f * n_x * n_y, c, th, tw)).astype('uint8')
    ref = opipe.stitch_mean_2d(tiles, f, (h, w), (th, tw), (n_x, n_y, xs, ys)).reshape(f, c, h, w)
    got = B.stitch_weighted_2d(tiles, f, (h, w), xs, ys, (th, tw), np.ones(th), np.ones(tw))
    assert np.array_equal(got, ref)


@pytest.mark.parametrize('h,w,th,tw,add,c', GRIDS_2D)
def test_constant_tiles_give_the_constant(h, w, th, tw, add, c):
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
    _, wh, ww = P.blend_tables((th, tw))
    for v in (0, 1, 128, 255):
        tiles = np.full((n_x * n_y, c, th, tw), v, np.uint8)
        assert np.all(B.stitch_weighted_2d(tiles, 1, (h, w), xs, ys, (th, tw), wh, ww) == v)
    vol, patch = (20, 40, 36), (8, 16, 16)
    n_z, n_x, n_y, zs, xs, ys = tiling.grid_3d(vol, patch, 2)
    tiles = np.full((n_z * n_x * n_y, 1, *patch), 255, np.uint8)
    assert np.all(B.stitch_weighted(tiles, 1, 1, vol, zs, xs, ys, patch, *P.blend_tables(patch)) == 255)


def test_single_cover_is_the_tile():
    """Where one tile covers a pixel, the result is that tile's value (tiles side by side, no overlap)."""
    n_x, n_y, xs, ys = tiling.grid_2d(64, 96, (32, 48), 0)
    tiles = np.random.default_rng(1).integers(0, 256, (n_x * n_y, 1, 32, 48)).astype('uint8')
    got = B.stitch_weighted_2d(tiles, 1, (64, 96), xs, ys, (32, 48), *P.blend_tables((32, 48))[1:])
    assert np.array_equal(got, opipe.stitch_mean_2d(tiles, 1, (64, 96), (32, 48), (n_x, n_y, xs, ys)).reshape(got.shape))


def test_blend_removes_the_tile_edge_step():
    """A 896-px row, 512-px tiles, add_tile=1 (starts 0, 192, 384): the first tile says 0, its neighbours 255. The mean
    stitch jumps by 127 between two adjacent pixels; the Gaussian blend changes by at most 4 per pixel."""
    n_x, n_y, xs, ys = tiling.grid_2d(16, 896, (16, 512), 1)
    assert n_x == 2 and list(ys) == [0, 192, 384]
    tiles = np.zeros((n_x * n_y, 1, 16, 512), np.uint8)
    tiles[[1, 2, 4, 5]] = 255                               # column tiles 1 and 2 of both tile rows
    mean = opipe.stitch_mean_2d(tiles, 1, (16, 896), (16, 512), (n_x, n_y, xs, ys)).reshape(16, 896)
    blend = B.stitch_weighted_2d(tiles, 1, (16, 896), xs, ys, (16, 512), *P.blend_tables((16, 512))[1:])[0, 0]
    assert np.abs(np.diff(mean.astype(int), axis=1)).max() == 127
    assert np.abs(np.diff(blend.astype(int), axis=1)).max() <= 4
    assert blend[0, 0] == 0 and blend[0, -1] == 255


@pytest.mark.parametrize('z,d,add,world', [(40, 8, 1, 2), (40, 8, 1, 3), (64, 16, 0, 4), (8, 8, 1, 2), (50, 16, 2, 8),
                                           (6, 8, 0, 2), (33, 8, 1, 5), (40, 8, 2, 1)] + _random_zslab_cases())
def test_zslab_local_weighted_stitch_equals_whole_volume(z, d, add, world):
    """Every rank (or z-row group) of tiling.zslab_plan stitches its own planes from its rows plus the borrowed ones,
    with starts relative to its first own plane (negative for rows that begin below it): the result equals the
    whole-volume weighted stitch, because the exact sums do not depend on which tiles are summed first."""
    x, y, h, w = 20, 24, 16, 16
    n_z, n_x, n_y, zs, xs, ys = tiling.grid_3d((z, x, y), (d, h, w), add)
    if z < d and n_z > 1:
        pytest.skip('the reference itself fails on undersized volumes split into several patches')
    rng = np.random.default_rng(z * 100 + world)
    patches = rng.integers(0, 256, (n_z * n_x * n_y, 1, d, h, w)).astype('uint8')
    tables = P.blend_tables((d, h, w))
    full = B.stitch_weighted(patches, 1, 1, (z, x, y), zs, xs, ys, (d, h, w), *tables)[0, 0]
    n_xy = n_x * n_y
    for p in tiling.zslab_plan(zs, d, z, world):
        lo, _ = p['rows']
        o0, o1 = p['own']
        if o1 <= o0:
            continue
        rows = list(range(*p['rows'])) + [zi for s in sorted(p['borrow']) for zi in p['borrow'][s]]
        local = patches[lo * n_xy:(lo + len(rows)) * n_xy]
        zs_local = [int(zs[zi]) - o0 for zi in rows]
        st = B.stitch_weighted(local, 1, 1, (o1 - o0, x, y), zs_local, xs, ys, (d, h, w), *tables)[0, 0]
        assert np.array_equal(st, full[o0:o1]), p


def test_blend_mode():
    assert P.blend_mode(None) is None
    assert P.blend_mode('gaussian') == 'gaussian'
    for bad in ('Gaussian', 'mean', 1, True, '', 'gauss'):
        with pytest.raises(ValueError):
            P.blend_mode(bad)


@pytest.mark.parametrize('bad', ['Gaussian', 'mean', 1, True])
def test_predictors_reject_bad_blend_before_any_engine(bad):
    """The checks run before a checkpoint is read or an Engine created, so they need neither a file nor a GPU."""
    from bio_image_unet_b200 import siam_unet, unet, unet3d
    img2d = np.zeros((1, 64, 64), np.uint8)
    cases = [
        lambda: unet.Predict(img2d, 'x.tif', 'missing.pt', resize_dim=(64, 64), blend=bad, show_progress=False,
                             device='cuda:0'),
        lambda: unet.Session('missing.pt', resize_dim=(64, 64), blend=bad),
        lambda: siam_unet.Predict(img2d, 'x.tif', 'missing.pt', resize_dim=(64, 64), blend=bad, show_progress=False,
                                  device='cuda:0'),
        lambda: siam_unet.Session('missing.pt', resize_dim=(64, 64), blend=bad),
        lambda: unet3d.Predict(np.zeros((8, 32, 32), np.uint8), 'x.tif', 'missing.pt', resize_dim=(8, 32, 32),
                               blend=bad, progress_bar=False, device='cuda:0'),
        lambda: unet3d.Session('missing.pt', (8, 32, 32), blend=bad),
    ]
    for make in cases:
        with pytest.raises(ValueError):
            make()
