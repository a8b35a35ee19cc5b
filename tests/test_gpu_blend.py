"""Gaussian overlap blending on the B200: the weighted-stitch kernel equals the numpy reference bit for bit, and every
predictor with blend='gaussian' writes exactly the weighted stitch of its own uint8 result tiles - across precisions,
twin-encoder forms, z-row groups, movie chunks, test-time augmentation and 2-rank sharding."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from bio_image_unet_b200 import engine as E
from bio_image_unet_b200 import pipeline2d as P
from bio_image_unet_b200 import tiff, tiling
from tests import _blend_ref as B
from tests.test_blend_host import GRIDS_2D
from tests.test_gpu_tta import _unet3d_ckpt, _unet_ckpt

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GRIDS_3D = [((20, 40, 36), (8, 16, 16)), ((6, 20, 12), (8, 16, 16)), ((17, 33, 40), (8, 32, 20))]


def _tables(kind, tile, rng):
    if kind == 'gauss':
        return P.blend_tables(tile)
    return tuple([int(v) for v in rng.integers(0, 1025, n)] for n in tile)


def _kernel(tiles, frames, channels, out_zhw, zs, ys, xs, tile, tables):
    got = E.stitch_weighted_u8(torch.from_numpy(tiles).to(DEV), frames, channels, out_zhw, zs, ys, xs, tile, *tables)
    return got.cpu().numpy()


# ---- 1. the kernel ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['gauss', 'random'])
@pytest.mark.parametrize('c', [1, 3])
@pytest.mark.parametrize('h,w,th,tw,add,_c', GRIDS_2D)
def test_kernel_2d_bit_exact(kind, c, h, w, th, tw, add, _c):
    rng = np.random.default_rng(h * w + add + c)
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
    f = 2
    tiles = rng.integers(0, 256, (f * n_x * n_y, c, th, tw)).astype('uint8')
    if kind == 'gauss':
        tables = P.blend_tables((th, tw))
    else:
        tables = ([1], *_tables('random', (th, tw), rng))
    want = B.stitch_weighted(tiles, f, c, (1, h, w), [0], xs, ys, (1, th, tw), *tables)
    assert np.array_equal(_kernel(tiles, f, c, (1, h, w), [0], xs, ys, (1, th, tw), tables), want)


@pytest.mark.parametrize('kind', ['gauss', 'random'])
@pytest.mark.parametrize('add', [0, 1, 2])
@pytest.mark.parametrize('vol,patch', GRIDS_3D)
def test_kernel_3d_bit_exact(kind, add, vol, patch):
    rng = np.random.default_rng(sum(vol) + add)
    n_z, n_x, n_y, zs, xs, ys = tiling.grid_3d(vol, patch, add)
    for c in (1, 2):
        tiles = rng.integers(0, 256, (n_z * n_x * n_y, c, *patch)).astype('uint8')
        tables = _tables(kind, patch, rng)
        want = B.stitch_weighted(tiles, 1, c, vol, zs, xs, ys, patch, *tables)
        assert np.array_equal(_kernel(tiles, 1, c, vol, zs, xs, ys, patch, tables), want)
        # starts relative to a later first plane, as the z-slab stitches pass them: negative for rows below it
        z0 = int(zs[-1]) // 2 + 1
        if z0 < vol[0]:
            local = [int(v) - z0 for v in zs]
            out = (vol[0] - z0, *vol[1:])
            want = B.stitch_weighted(tiles, 1, c, out, local, xs, ys, patch, *tables)
            assert np.array_equal(_kernel(tiles, 1, c, out, local, xs, ys, patch, tables), want)


@pytest.mark.parametrize('h,w,th,tw,add,c', GRIDS_2D)
def test_unit_tables_equal_stitch_mean(h, w, th, tw, add, c):
    rng = np.random.default_rng(7 + add)
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
    tiles = torch.from_numpy(rng.integers(0, 256, (2 * n_x * n_y, c, th, tw)).astype('uint8')).to(DEV)
    mean = E.stitch_mean_u8(tiles, 2, c, (h, w), xs, ys, (th, tw))
    got = E.stitch_weighted_u8(tiles, 2, c, (1, h, w), [0], xs, ys, (1, th, tw), [1], [1] * th, [1] * tw)
    assert torch.equal(got.view(2, c, h, w), mean)


def test_extremes_do_not_overflow():
    """All values 255, all weights 1024: every product and sum is at its largest (the 3D grid with add_patch 2 has the
    densest overlap of the grids above). The result is 255 everywhere."""
    vol, patch = GRIDS_3D[0][0], GRIDS_3D[0][1]
    n_z, n_x, n_y, zs, xs, ys = tiling.grid_3d(vol, patch, 2)
    tiles = np.full((n_z * n_x * n_y, 1, *patch), 255, np.uint8)
    tables = tuple([1024] * n for n in patch)
    assert np.all(_kernel(tiles, 1, 1, vol, zs, xs, ys, patch, tables) == 255)
    h, w, th, tw, add, _ = GRIDS_2D[4]
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, (th, tw), add)
    tiles = np.full((n_x * n_y, 1, th, tw), 255, np.uint8)
    assert np.all(_kernel(tiles, 1, 1, (1, h, w), [0], xs, ys, (1, th, tw), ([1024], [1024] * th, [1024] * tw)) == 255)


def test_bad_tables_are_rejected():
    tiles = torch.zeros((1, 1, 16, 16), dtype=torch.uint8, device=DEV)
    with pytest.raises(ValueError):
        E.stitch_weighted_u8(tiles, 1, 1, (1, 16, 16), [0], [0], [0], (1, 16, 16), [1], [1] * 15, [1] * 16)
    with pytest.raises(ValueError):
        E.stitch_weighted_u8(tiles, 1, 1, (1, 16, 16), [0], [0], [0], (1, 16, 16), [1], [1025] * 16, [1] * 16)


# ---- 2. every predictor writes the weighted stitch of its own result tiles ------------------------------------------
def _tif(path):
    return tiff.imread(str(path))


@pytest.mark.parametrize('network,precision', [('Unet', 'bf16'), ('Unet', 'fp16'), ('Unet', 'tf32'), ('Unet', 'fp32'),
                                               ('AttentionUnet', 'bf16'), ('Unet_v0', 'bf16')])
def test_unet_predict(tmp_path, network, precision):
    from bio_image_unet_b200.unet import Predict
    ck = tmp_path / 'u.pt'
    torch.save(_unet_ckpt(network), ck)
    imgs = np.random.default_rng(5).integers(0, 3000, (3, 90, 77)).astype(np.uint16)
    rd = (64, 64)
    p = Predict(imgs.copy(), str(tmp_path / 'b.tif'), str(ck), network=network, resize_dim=rd, add_tile=1,
                show_progress=False, device=DEV, precision=precision, keep_intermediates=True, blend='gaussian')
    want = B.stitch_weighted_2d(p.result_patches, 3, (90, 77), p.X_start, p.Y_start, rd, *P.blend_tables(rd)[1:])
    assert np.array_equal(_tif(tmp_path / 'b.tif'), np.squeeze(want).astype(np.float16))


@pytest.mark.parametrize('mode,norm', [('concat', 'single'), ('concat', 'first'), ('control', 'single')])
def test_siam_predict(tmp_path, mode, norm):
    from bio_image_unet_b200.siam_unet import Predict
    from bio_image_unet_b200.siam_unet.siam_unet import Siam_UNet
    torch.manual_seed(2)
    ck = tmp_path / 's.pt'
    torch.save({'state_dict': Siam_UNet(n_filter=8, mode=mode).eval().state_dict(), 'n_filter': 8, 'mode': mode}, ck)
    movie = np.random.default_rng(4).integers(0, 2000, (5, 40, 52)).astype(np.uint16)
    rd = (32, 32)
    p = Predict(movie, str(tmp_path / 'b.tif'), str(ck), resize_dim=rd, add_tile=1, normalization_mode=norm,
                show_progress=False, device=DEV, precision='bf16', keep_intermediates=True, workspace_gb=0.02,
                blend='gaussian')
    res = p.result_patches.reshape(-1, 1, *rd)
    want = B.stitch_weighted_2d(res, 5, (40, 52), p.X_start, p.Y_start, rd, *P.blend_tables(rd)[1:])
    assert np.array_equal(_tif(tmp_path / 'b.tif'), want[:, 0])


@pytest.mark.parametrize('add_patch', [0, 1])
def test_unet3d_predict(tmp_path, add_patch):
    from bio_image_unet_b200.unet3d import Predict
    ck = tmp_path / 'v.pt'
    torch.save(_unet3d_ckpt(), ck)
    vol = np.random.default_rng(11).integers(0, 3000, (30, 40, 36)).astype('uint16')
    rd = (8, 16, 16)
    p = Predict(vol.copy(), str(tmp_path / 'b.tif'), str(ck), resize_dim=rd, add_patch=add_patch, progress_bar=False,
                device=DEV, precision='bf16', keep_intermediates=True, workspace_gb=0.01, blend='gaussian')
    want = B.stitch_weighted(p.result_patches, 1, 1, vol.shape, p.Z_start, p.X_start, p.Y_start, rd,
                             *P.blend_tables(rd))
    assert np.array_equal(_tif(tmp_path / 'b.tif'), want[0, 0].astype(np.float16))


def test_no_overlap_is_unchanged(tmp_path):
    """Tiles side by side: every pixel has one covering tile, so the blend returns the reference's result."""
    from bio_image_unet_b200.siam_unet import Predict as PredictSiam
    from bio_image_unet_b200.siam_unet.siam_unet import Siam_UNet
    from bio_image_unet_b200.unet import Session
    from bio_image_unet_b200.unet3d import Session as Session3D
    frames = torch.from_numpy(np.random.default_rng(3).integers(0, 3000, (2, 128, 192)).astype(np.uint16)).to(DEV)
    outs = []
    for blend in (None, 'gaussian'):
        ses = Session(_unet_ckpt(), resize_dim=(64, 64), device=DEV, precision='bf16', blend=blend)
        outs.append(ses.predict_device(frames))
        ses.close()
    assert torch.equal(outs[0], outs[1])
    vol = np.random.default_rng(6).integers(0, 3000, (16, 32, 48)).astype('uint16')
    outs = []
    for blend in (None, 'gaussian'):
        ses = Session3D(_unet3d_ckpt(), (8, 16, 16), device=DEV, precision='bf16', blend=blend)
        outs.append(ses.predict(vol.copy(), to_host=False).cpu())
        ses.close()
    assert torch.equal(outs[0], outs[1])
    torch.manual_seed(2)
    ck = tmp_path / 's.pt'
    torch.save({'state_dict': Siam_UNet(n_filter=8, mode='concat').eval().state_dict(), 'n_filter': 8,
                'mode': 'concat'}, ck)
    movie = np.random.default_rng(4).integers(0, 2000, (3, 32, 48)).astype(np.uint16)
    for blend in (None, 'gaussian'):                          # resize_dim=None: one tile per frame
        PredictSiam(movie, str(tmp_path / f'{blend}.tif'), str(ck), resize_dim=None, show_progress=False, device=DEV,
                    precision='bf16', blend=blend)
    assert np.array_equal(_tif(tmp_path / 'None.tif'), _tif(tmp_path / 'gaussian.tif'))


# ---- 3. composition with tta, z-row groups, movie chunks -------------------------------------------------------------
def test_tta_and_blend_compose():
    from bio_image_unet_b200.unet import Session
    from bio_image_unet_b200.unet3d import Session as Session3D
    frames = torch.from_numpy(np.random.default_rng(1).integers(0, 3000, (3, 100, 90)).astype(np.uint16)).to(DEV)
    rd = (64, 64)
    ses = Session(_unet_ckpt(), resize_dim=rd, add_tile=1, device=DEV, precision='bf16', tta='flips', blend='gaussian')
    got = ses.predict_device(frames, keep=True)
    _, _, xs, ys = ses.last['grid']
    want = E.stitch_weighted_u8(ses.last['result_tiles'], 3, 1, (1, 100, 90), [0], xs, ys, (1, *rd), *P.blend_tables(rd))
    assert torch.equal(got, want.view(got.shape))
    base = Session(_unet_ckpt(), resize_dim=rd, add_tile=1, device=DEV, precision='bf16', tta='flips')
    base.predict_device(frames, keep=True)
    assert torch.equal(ses.last['result_tiles'], base.last['result_tiles'])     # the same TTA mean tiles
    ses.close()
    base.close()
    vol = np.random.default_rng(11).integers(0, 3000, (30, 40, 36)).astype('uint16')
    rd3 = (8, 16, 16)
    ses = Session3D(_unet3d_ckpt(), rd3, add_patch=1, device=DEV, precision='bf16', tta='flips', blend='gaussian',
                    workspace_gb=0.01)
    got = ses.predict(vol.copy(), keep=True, to_host=False).cpu().numpy()
    want = B.stitch_weighted(ses.result_patches, 1, 1, vol.shape, ses.Z_start, ses.X_start, ses.Y_start, rd3,
                             *P.blend_tables(rd3))
    assert np.array_equal(got, want[0, 0])
    ses.close()


@pytest.mark.parametrize('add_patch', [0, 1])
def test_unet3d_groups_equal_whole_volume(add_patch):
    from bio_image_unet_b200.unet3d import Session
    vol = np.random.default_rng(12).integers(0, 3000, (44, 40, 48)).astype('uint16')
    ses = Session(_unet3d_ckpt(), (8, 16, 16), add_patch=add_patch, device=DEV, precision='bf16', blend='gaussian',
                  workspace_gb=0.01)
    piped = ses.predict(vol.copy()).copy()                     # z-row groups, stitched group by group
    assert ses.N_z >= 4
    whole = ses.predict(vol.copy(), to_host=False).cpu().numpy()
    assert np.array_equal(piped, whole)
    ses.close()


def test_predict_movie_chunks_equal_one_chunk():
    from bio_image_unet_b200.unet import Session
    frames = np.random.default_rng(8).integers(0, 3000, (5, 100, 90)).astype(np.uint16)
    ses = Session(_unet_ckpt(), resize_dim=(64, 64), add_tile=1, device=DEV, precision='bf16', blend='gaussian')
    one = ses.predict_movie(frames, chunk_frames=5)[0].copy()
    for chunk in (1, 2):
        assert np.array_equal(ses.predict_movie(frames, chunk_frames=chunk)[0], one), chunk
    ses.close()


# ---- 4. distributed ----------------------------------------------------------------------------------------------
def test_distributed_blend_matches_single_process(tmp_path):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29537', os.path.join(ROOT, 'tests', 'run_dist_blend.py'), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-3000:])
    assert r.returncode == 0
    assert os.path.exists(tmp_path / 'DIST_OK')
