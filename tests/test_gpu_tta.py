"""Test-time augmentation on the B200: the transform-taking gathers and the merge are bit-exact against torch
transforms, and every predictor's tta result equals the explicit composition plain gather -> torch T_t -> forward on
the same plan -> torch T_t^-1 -> ordered fp32 sum -> quantise -> the existing stitch, bit for bit."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from bio_image_unet_b200 import engine as E
from bio_image_unet_b200 import pipeline2d as P
from bio_image_unet_b200 import tiling
from tests.test_tta_host import T, T_inv

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PRECISIONS = ['bf16', 'fp16', 'tf32', 'fp32']


def _u8_of_mean(acc, k):
    return ((acc * (1.0 / k)) * 255).to(torch.uint8)


# ---- 1. gathers ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('src_kind', ['u8', 'lut_u8', 'lut_u16', 'f32'])
@pytest.mark.parametrize('shape,tile,add', [((45, 61), (32, 32), 1), ((20, 20), (20, 20), 0), ((13, 17), (16, 16), 0),
                                            ((70, 50), (48, 48), 1), ((9, 30), (12, 12), 1)])
@pytest.mark.parametrize('pad_mode', [0, 1])
def test_gather_2d_bit_exact(src_kind, shape, tile, add, pad_mode):
    if src_kind == 'f32' and pad_mode == 1:
        pytest.skip('the float32 gather pads by reflection only')
    g = torch.Generator().manual_seed(sum(shape) + add)
    h, w = shape
    f = 2
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, tile, add)
    if src_kind == 'u8':
        src = torch.randint(0, 256, (f, 1, h, w), generator=g, dtype=torch.uint8).to(DEV)
        lut = None
    elif src_kind == 'f32':
        src = torch.rand((f, 1, h, w), generator=g).to(DEV)
    else:
        hi = 256 if src_kind == 'lut_u8' else 65536
        src = torch.randint(0, hi, (f, 1, h, w), generator=g, dtype=torch.int32).to(
            torch.uint8 if hi == 256 else torch.uint16).to(DEV)
        lut = torch.randint(0, 256, (f, 65536), generator=g, dtype=torch.uint8).to(DEV)
    t1 = (1,) + tuple(tile)
    if src_kind == 'f32':
        plain = E.gather_tiles_f32(src, [0], xs, ys, t1)
    elif lut is None:
        plain = E.gather_tiles(src, [0], xs, ys, t1, pad_mode)
    else:
        plain = E.gather_tiles_lut(src, lut, [0], xs, ys, t1, pad_mode)
    for t in range(8 if tile[0] == tile[1] else 4):
        if src_kind == 'f32':
            got = E.gather_tiles_f32_tta(src, [0], xs, ys, t1, 2, t)
        else:
            got = E.gather_tiles_tta(src, [0], xs, ys, t1, pad_mode, 2, t, lut=lut)
        assert torch.equal(got, T(plain, 2, t).contiguous()), t


@pytest.mark.parametrize('src_kind', ['lut_u16', 'u8', 'f32'])
@pytest.mark.parametrize('vol,patch,add', [((20, 40, 36), (8, 16, 16), 1), ((6, 20, 12), (8, 16, 16), 0),
                                           ((17, 33, 40), (8, 32, 20), 1)])
def test_gather_3d_bit_exact(src_kind, vol, patch, add):
    g = torch.Generator().manual_seed(sum(vol))
    if src_kind == 'f32':
        pz = tuple(min(a, b) for a, b in zip(vol, patch))
        zs, ys, xs = (tiling.strided_starts(vol[i], pz[i], 0.3) for i in range(3))
        src = torch.rand((1, *vol), generator=g).to(DEV)
        plain = E.gather_tiles_f32(src, zs, ys, xs, pz)
        for t in range(8):
            assert torch.equal(E.gather_tiles_f32_tta(src, zs, ys, xs, pz, 3, t), T(plain, 3, t).contiguous()), t
        return
    _, _, _, zs, ys, xs = tiling.grid_3d(vol, patch, add)
    if src_kind == 'u8':
        src = torch.randint(0, 256, (1, *vol), generator=g, dtype=torch.uint8).to(DEV)
        lut = None
        plain = E.gather_tiles(src, zs, ys, xs, patch, 0)
    else:
        src = torch.randint(0, 65536, (1, *vol), generator=g, dtype=torch.int32).to(torch.uint16).to(DEV)
        lut = torch.randint(0, 256, (1, 65536), generator=g, dtype=torch.uint8).to(DEV)
        plain = E.gather_tiles_lut(src, lut, zs, ys, xs, patch, 0)
    for t in range(8):
        got = E.gather_tiles_tta(src, zs, ys, xs, patch, 0, 3, t, lut=lut)
        assert torch.equal(got, T(plain, 3, t).contiguous()), t


def test_gather_rejects_transposed_non_square():
    src = torch.zeros((1, 1, 32, 64), dtype=torch.uint8, device=DEV)
    with pytest.raises(E._lib.BiuError):
        E.gather_tiles_tta(src, [0], [0], [0], (1, 32, 64), 0, 2, 4)


# ---- 2. merge --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('dims,shape,k', [(2, (5, 2, 48, 48), 8), (2, (3, 1, 20, 20), 8), (2, (4, 3, 32, 64), 4),
                                          (3, (3, 2, 8, 16, 24), 8), (2, (2, 1, 16, 16), 1)])
def test_accumulate_bit_exact(dims, shape, k):
    g = torch.Generator().manual_seed(k + len(shape))
    vals = [torch.rand(shape, generator=g).to(DEV) for _ in range(k)]
    acc = torch.empty(shape, dtype=torch.float32, device=DEV)
    out_u8 = torch.empty(shape, dtype=torch.uint8, device=DEV)
    out_f = torch.empty(shape, dtype=torch.float32, device=DEV)
    ref = None
    for p in range(k):
        E.tta_accumulate(vals[p], acc, dims, p, p, k, out_u8=out_u8, out_f32=out_f)
        v = T_inv(vals[p], dims, p)
        ref = v if ref is None else ref + v
    mean = ref * (1.0 / k)
    assert torch.equal(out_f, mean)
    assert torch.equal(out_u8, _u8_of_mean(ref, k))


def _unet_ckpt(network='Unet', n_filter=8, seed=0):
    from bio_image_unet_b200.unet import AttentionUnet, Unet, Unet_v0
    cls = {'Unet': Unet, 'AttentionUnet': AttentionUnet, 'Unet_v0': Unet_v0}[network]
    torch.manual_seed(seed)
    m = cls(n_filter=n_filter).eval()
    return {'state_dict': m.state_dict(), 'n_filter': n_filter, 'in_channels': 1, 'out_channels': 1}


def test_accumulate_k1_equals_engine_u8():
    from bio_image_unet_b200.unet import Session
    ses = Session(_unet_ckpt(), resize_dim=(64, 64), device=DEV, precision='bf16')
    ses._ensure_plan(6)
    tiles = torch.randint(0, 256, (6, 1, 64, 64), dtype=torch.uint8, device=DEV)
    val, u8 = ses.engine.forward(tiles, want_val=True, want_u8=True)
    out = torch.empty_like(u8)
    E.tta_accumulate(val, None, 2, 0, 0, 1, out_u8=out)
    assert torch.equal(out, u8)
    ses.close()


# ---- 3. every predictor decomposes exactly -------------------------------------------------------------------
def _compose(eng, tiles, tile_batch, codes, dims, prev=None):
    """sum over t of T_t^-1(forward(T_t(tiles))) in ascending t, fp32, on the plan the predictor used."""
    acc = None
    for t in codes:
        tt = T(tiles, dims, t).contiguous()
        pt = None if prev is None else T(prev, dims, t).contiguous()
        _, val = P.run_tiles(eng, tt, tile_batch, prev_tiles=pt, want_val=True)
        v = T_inv(val, dims, t)
        acc = v if acc is None else acc + v
    return acc


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('network,tta', [('Unet', 'flips'), ('Unet', 'dihedral'), ('AttentionUnet', 'dihedral'),
                                         ('Unet_v0', 'flips')])
def test_unet_decomposes(precision, network, tta):
    from bio_image_unet_b200.unet import Session
    rd, add = (64, 64), 1
    ses = Session(_unet_ckpt(network), resize_dim=rd, add_tile=add, device=DEV, precision=precision, network=network,
                  tta=tta)
    # a budget of 10 tiles: several forwards per pass
    ses._planner.workspace_bytes = 10 * (ses.engine.plan(1, rd) + P.tta_extra_bytes(tta, 1, rd))
    frames = torch.from_numpy(np.random.default_rng(1).integers(0, 3000, (3, 100, 90)).astype(np.uint16)).to(DEV)
    got = ses.predict_device(frames)
    f, h, w = frames.shape
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, rd, add)
    tiles = E.gather_tiles_lut(frames.view(f, 1, h, w), ses.lut_device(frames), [0], xs, ys, (1, *rd), 0)
    codes = P.tta_codes(tta, 2, rd)
    acc = _compose(ses.engine, tiles, ses.tile_batch, codes, 2)
    want = E.stitch_mean_u8(_u8_of_mean(acc, len(codes)), f, 1, (h, w), xs, ys, rd)
    assert ses.tile_batch < f * n_x * n_y          # several forwards per pass
    assert torch.equal(got, want)
    ses.close()


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('siam_path', ['shared_encoder', 'two_input'])
def test_siam_decomposes(precision, siam_path):
    """Both Siam_UNet paths: the shared twin encoder ('concat' in 'single' mode, batches of unique tiles through
    run_tiles with n_per) and the two-input network ('control')."""
    from bio_image_unet_b200.siam_unet import Session
    from bio_image_unet_b200.siam_unet.siam_unet import Siam_UNet
    shared = siam_path == 'shared_encoder'
    torch.manual_seed(2)
    mode = 'concat' if shared else 'control'
    ck = {'state_dict': Siam_UNet(n_filter=8, mode=mode).eval().state_dict(), 'n_filter': 8, 'mode': mode}
    rd = (32, 32)
    ses = Session(ck, resize_dim=rd, add_tile=1, device=DEV, precision=precision, tta='dihedral', workspace_gb=0.02)
    assert ses.shared_encoder == shared
    movie = torch.from_numpy(np.random.default_rng(4).integers(0, 2000, (5, 40, 52)).astype(np.uint16))
    n_pairs = 4
    needed, p_pos, c_pos = ses.chunk_frames(5, 1, 5)
    frames = movie[needed].contiguous().to(DEV)
    p_sel, c_sel = E._dev_i64(p_pos, DEV), E._dev_i64(c_pos, DEV)
    k, h, w = frames.shape
    _, n_x, n_y, xs, ys = ses.grid(h, w)
    ses._ensure_plan(rd, n_pairs * n_x * n_y, n_x * n_y if shared else 0)
    got = ses.predict_pairs_device(frames, p_sel, c_sel)
    codes = list(range(8))
    hist = E.histogram(frames)
    lut, _ = E.norm_lut(hist, hist, k, ses.clip_threshold[0], ses.clip_threshold[1], False)
    if shared:
        tiles_u = E.gather_tiles_lut(frames.view(k, 1, h, w), lut, [0], xs, ys, (1, *rd), 1)
        n_per = n_x * n_y
        acc = None
        for t in codes:
            vals = []
            P.run_tiles(ses.engine, T(tiles_u, 2, t).contiguous(), ses.tile_batch, n_per=n_per,
                        on_val=lambda s, v: vals.append(v.clone()))
            v = T_inv(torch.cat(vals), 2, t)
            acc = v if acc is None else acc + v
    else:
        norm = E.apply_lut(frames, lut)
        cur = E.gather_tiles(norm[c_sel].contiguous().view(n_pairs, 1, h, w), [0], xs, ys, (1, *rd), 1)
        prev = E.gather_tiles(norm[p_sel].contiguous().view(n_pairs, 1, h, w), [0], xs, ys, (1, *rd), 1)
        acc = _compose(ses.engine, cur, ses.tile_batch, codes, 2, prev=prev)
    want = E.stitch_mean_u8(_u8_of_mean(acc, 8), n_pairs, 1, (h, w), xs, ys, rd)
    assert torch.equal(got, want)
    ses.close()


def _unet3d_ckpt(seed=5):
    from bio_image_unet_b200.unet3d import UNet3D
    torch.manual_seed(seed)
    return {'state_dict': UNet3D(n_filter=4).eval().state_dict(), 'n_filter': 4, 'in_channels': 1, 'out_channels': 1}


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('add_patch', [0, 1])
def test_unet3d_decomposes(precision, add_patch):
    from bio_image_unet_b200.unet3d import Session
    rd = (8, 16, 16)
    vol = np.random.default_rng(11).integers(0, 3000, (30, 40, 36)).astype('uint16')
    ses = Session(_unet3d_ckpt(), rd, add_patch=add_patch, device=DEV, precision=precision, tta='flips',
                  workspace_gb=0.01)
    piped = ses.predict(vol.copy())                            # grouped (pipelined) path: N_z >= 2
    whole = ses.predict(vol.copy(), to_host=False).cpu().numpy()
    assert ses.N_z >= 2
    z, x, y = vol.shape
    src = torch.from_numpy(vol).to(DEV).view(1, z, x, y)
    total = E.hist_sum(E.histogram(src.view(z, x, y).contiguous()))
    lut, _ = E.norm_lut(total, total, 1, 0., 99.8, False)
    zs = [int(v) for v in ses.Z_start]
    patches = E.gather_tiles_lut(src, lut, zs, ses.X_start, ses.Y_start, rd, 0)
    n = patches.shape[0]
    acc = _compose(ses.engine, patches.reshape(n, 1, *rd), ses.tile_batch, range(8), 3)
    want = E.stitch_mod3_u8(_u8_of_mean(acc, 8).reshape(n, *rd), (z, x, y), zs, ses.X_start, ses.Y_start, rd)
    assert np.array_equal(whole, want.cpu().numpy())
    assert np.array_equal(piped, whole)
    ses.close()


@pytest.mark.parametrize('precision', PRECISIONS)
def test_mo3d_decomposes(precision):
    from bio_image_unet_b200.multi_output_unet3d import Session
    from bio_image_unet_b200.multi_output_unet3d.multi_output_unet3d import MultiOutputUnet3D
    heads = {'a': {'channels': 1, 'activation': 'sigmoid'}, 'b': {'channels': 2, 'activation': None}}
    torch.manual_seed(3)
    m = MultiOutputUnet3D(output_heads=heads, n_filter=4, use_interpolation=True).eval()
    ck = {'state_dict': m.state_dict(), 'n_filter': 4, 'in_channels': 1, 'output_heads': heads, 'use_interpolation': True}
    ses = Session(ck, max_patch_size=(8, 32, 32), overlap_factor=0.25, device=DEV, precision=precision, tta='flips',
                  workspace_gb=0.02)
    imgs = np.random.default_rng(6).integers(0, 3000, (2, 12, 40, 48)).astype('uint16')
    got = ses.predict(imgs, to_host=False)
    vols = torch.from_numpy(imgs).to(DEV)
    norm = ses._normalise(vols, 0)
    patches = E.gather_tiles_f32(norm, ses.Z_start, ses.Y_start, ses.X_start, ses.patch_size)
    n = patches.shape[0]
    acc = _compose(ses.engine, patches.reshape(n, 1, *ses.patch_size), ses.tile_batch, range(8), 3)
    # predict() chunks volumes: stitch chunk-wise exactly as it does (the ramp blend is per volume)
    want = E.stitch_ramp_f32((acc * 0.125).contiguous(), 2, 3, imgs.shape[1:], ses.Z_start, ses.Y_start, ses.X_start,
                             ses.patch_size, 16)
    assert torch.equal(got, want)
    ses.close()


@pytest.mark.parametrize('precision', PRECISIONS)
@pytest.mark.parametrize('tta', ['flips', 'dihedral'])
def test_mo2d_decomposes(precision, tta):
    from bio_image_unet_b200.multi_output_unet import Predict
    from bio_image_unet_b200.multi_output_unet.multi_output_unet import MultiOutputUnet
    heads = {'m': {'channels': 1, 'activation': 'sigmoid'}, 'd': {'channels': 1, 'activation': None}}
    torch.manual_seed(8)
    m = MultiOutputUnet(output_heads=heads, n_filter=8).eval()
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        ckpt = os.path.join(d, 'mo2d.pt')
        torch.save({'state_dict': m.state_dict(), 'n_filter': 8, 'in_channels': 1, 'output_heads': heads}, ckpt)
        imgs = np.random.default_rng(9).integers(0, 4000, (2, 70, 70)).astype('uint16')
        kw = dict(network='MultiOutputUnet', max_patch_size=(48, 48), show_progress=False, device=DEV,
                  precision=precision, keep_intermediates=True)
        p = Predict(imgs.copy(), ckpt, tta=tta, **kw)
        base = Predict(imgs.copy(), ckpt, **kw)
    eng = E.Engine('mo2d', m.state_dict(), 8, 1, [(k, 1, heads[k]['activation']) for k in heads], precision=precision,
                   device=DEV)
    patches = torch.from_numpy(base.patches).to(DEV)[:, None]
    tb = P.pick_tile_batch(eng, (48, 48), patches.shape[0], int(24.0 * 2 ** 30))
    codes = P.tta_codes(tta, 2, (48, 48))
    mean = _compose(eng, patches, tb, codes, 2) * (1.0 / len(codes))
    assert np.array_equal(p.result_patches, mean.cpu().numpy())
    t, h, w = imgs.shape
    idx = (np.arange(t)[:, None, None] * p.N_per_img + np.arange(p.N_x)[None, :, None] * p.N_y +
           np.arange(p.N_y)[None, None, :]).astype(np.int32)
    for c, key in enumerate(heads):
        tiles_k = mean[:, c:c + 1].contiguous()
        fill = tiles_k.to(torch.float16).float().mean().to(torch.float16).float().reshape(1)
        st = E.stitch_margin_f32(tiles_k, torch.from_numpy(idx).to(DEV), t, 1, (max(48, h), max(48, w)), p.X_start,
                                 p.Y_start, (48, 48), fill, 20)
        assert np.array_equal(p.result[key], np.squeeze(st[:, :, :h, :w].cpu().numpy())), key
    eng.close()


# ---- 5. equivariance, 6. tta=None ------------------------------------------------------------------------------
@pytest.mark.parametrize('tta', ['flips', 'dihedral'])
def test_single_tile_equivariance(tta):
    from bio_image_unet_b200.unet import Session
    ses = Session(_unet_ckpt(seed=4), resize_dim=(64, 64), device=DEV, precision='bf16', tta=tta)
    x = torch.from_numpy(np.random.default_rng(2).integers(0, 255, (1, 64, 64)).astype(np.uint8)).to(DEV)
    base = ses.predict_device(x)[0, 0]
    for t in P.tta_codes(tta, 2, (64, 64)):
        y = ses.predict_device(T(x, 2, t).contiguous())[0, 0]
        d = (y.int() - T(base, 2, t).int()).abs().max().item()
        assert d <= 1, (t, d)
    ses.close()


def test_tta_none_is_byte_identical(tmp_path):
    from bio_image_unet_b200 import tiff
    from bio_image_unet_b200.unet import Predict
    ck = tmp_path / 'u.pt'
    torch.save(_unet_ckpt(), ck)
    imgs = np.random.default_rng(5).integers(0, 3000, (3, 90, 77)).astype(np.uint16)
    kw = dict(resize_dim=(64, 64), add_tile=1, show_progress=False, device=DEV, precision='bf16')
    Predict(imgs.copy(), str(tmp_path / 'a.tif'), str(ck), **kw)
    Predict(imgs.copy(), str(tmp_path / 'b.tif'), str(ck), tta=None, **kw)
    assert np.array_equal(tiff.imread(str(tmp_path / 'a.tif')), tiff.imread(str(tmp_path / 'b.tif')))


# ---- 4. parity against the CPU oracle on the stress net ---------------------------------------------------------
def test_oracle_tta_parity():
    from tests import _golden
    from tests.test_tta_host import oracle_tta_unet
    from bio_image_unet_b200.unet import Session
    g = _golden.load('unet_single')
    assert str(g['mode']) == 'single' and not bool(g['invert'])
    sd = _golden.state_dict(g)
    rd = tuple(int(v) for v in g['resize_dim'])
    imgs = g['imgs'][:2].copy()
    want = oracle_tta_unet(imgs, sd, P.tta_codes('flips', 2, rd), rd, int(g['add_tile']), clip_threshold=tuple(g['clip']))
    ses = Session({'state_dict': sd, 'n_filter': int(g['n_filter']), 'in_channels': 1, 'out_channels': 1},
                  resize_dim=rd, add_tile=int(g['add_tile']), clip_threshold=tuple(g['clip']), device=DEV,
                  precision='fp32', tta='flips')
    got = ses.predict_device(torch.from_numpy(np.ascontiguousarray(imgs)).to(DEV)).cpu().numpy()
    assert np.abs(got.astype(np.int16) - want.reshape(got.shape).astype(np.int16)).max() <= 1
    ses.close()


# ---- 7. distributed ----------------------------------------------------------------------------------------------
def test_distributed_tta_matches_single_process(tmp_path):
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29533', os.path.join(ROOT, 'tests', 'run_dist_tta.py'), str(tmp_path)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    print(r.stdout[-3000:], r.stderr[-3000:])
    assert r.returncode == 0
    assert os.path.exists(tmp_path / 'DIST_OK')
