"""Test-time augmentation without a GPU: the transform table, its inverses, the `tta` argument checks of every
predictor, and an oracle-side TTA (the CPU reference functions with torch flips) that the GPU tests compare with."""
import numpy as np
import pytest
import torch

from bio_image_unet_b200 import pipeline2d as P
from oracle import models as omodels
from oracle import pipeline as opipe


# ---- the transform table: T_t(a) = a.flip(dims) [.transpose(-2, -1) when 2D bit 2 is set]; T_t^-1 in reverse order ----
def flip_dims(dims, t):
    return [d for bit, d in ((0, -1), (1, -2), (2, -3)) if (t >> bit) & 1 and not (dims == 2 and bit == 2)]


def T(a, dims, t):
    fd = flip_dims(dims, t)
    a = a.flip(fd) if fd else a
    return a.transpose(-2, -1) if dims == 2 and t & 4 else a


def T_inv(a, dims, t):
    a = a.transpose(-2, -1) if dims == 2 and t & 4 else a
    fd = flip_dims(dims, t)
    return a.flip(fd) if fd else a


def oracle_tta_unet(imgs, sd, codes, resize_dim, add_tile=0, network='Unet', clip_threshold=(0., 99.8)):
    """unet.Predict with test-time augmentation on the CPU oracle: the reference's normalisation, split and stitch,
    the fp32 forward on T_t of every patch, T_t^-1, an fp32 sum in ascending t, * (1 / K), (mean * 255) -> uint8."""
    shape = imgs.shape
    norm = opipe.preprocess_stack(imgs.copy(), 'single', clip_threshold, False)
    patches, grid = opipe.split_2d(norm, resize_dim, add_tile)
    x = torch.from_numpy(patches.astype('float32') / 255)
    acc = None
    with torch.no_grad():
        for t in codes:
            v = T_inv(omodels.FORWARD_2D[network](opipe._to_sd(sd), T(x, 2, t).contiguous())[0], 2, t)
            acc = v if acc is None else acc + v
    mean = acc * (1.0 / len(codes))
    res = (mean.numpy() * 255).astype('uint8')
    return opipe.stitch_mean_2d(res, shape[0], shape[1:], resize_dim, grid)


def test_transform_table_matches_numpy_compositions():
    a = np.arange(5 * 6, dtype=np.int32).reshape(5, 6)
    sq = np.arange(6 * 6, dtype=np.int32).reshape(6, 6)
    ta = torch.from_numpy(a)
    assert np.array_equal(T(ta, 2, 0).numpy(), a)
    assert np.array_equal(T(ta, 2, 1).numpy(), np.flip(a, 1))
    assert np.array_equal(T(ta, 2, 2).numpy(), np.flip(a, 0))
    assert np.array_equal(T(ta, 2, 3).numpy(), np.rot90(a, 2))
    ts = torch.from_numpy(sq)
    assert np.array_equal(T(ts, 2, 4).numpy(), sq.T)
    assert np.array_equal(T(ts, 2, 5).numpy(), np.rot90(sq, 1))          # flip x, then transpose
    assert np.array_equal(T(ts, 2, 6).numpy(), np.rot90(sq, -1))         # flip y, then transpose
    assert np.array_equal(T(ts, 2, 7).numpy(), np.rot90(sq, 2).T)        # anti-transpose
    v = np.arange(3 * 4 * 5).reshape(3, 4, 5)
    for t in range(8):
        ref = v
        for bit, ax in ((0, 2), (1, 1), (2, 0)):
            if (t >> bit) & 1:
                ref = np.flip(ref, ax)
        assert np.array_equal(T(torch.from_numpy(v), 3, t).numpy(), ref), t


@pytest.mark.parametrize('dims', [2, 3])
def test_inverse_undoes_and_codes_are_distinct(dims):
    shape = (2, 7, 7) if dims == 2 else (2, 3, 5, 7)
    a = torch.arange(int(np.prod(shape)), dtype=torch.float32).reshape(shape)
    seen = set()
    for t in range(8):
        b = T(a, dims, t)
        assert torch.equal(T_inv(b, dims, t), a)
        seen.add(b.numpy().tobytes())
    assert len(seen) == 8


def test_tta_codes():
    assert P.tta_codes(None, 2, (64, 64)) is None
    assert P.tta_codes('flips', 2, (32, 64)) == [0, 1, 2, 3]
    assert P.tta_codes('dihedral', 2, (64, 64)) == list(range(8))
    assert P.tta_codes('flips', 3, (8, 16, 32)) == list(range(8))
    for bad, dims, tile in (('dihedral', 2, (32, 64)), ('dihedral', 3, (16, 16, 16)), ('rot90', 2, (64, 64)),
                            ('', 2, (64, 64)), (True, 2, (64, 64)), ('Flips', 3, (8, 8, 8))):
        with pytest.raises(ValueError):
            P.tta_codes(bad, dims, tile)


def test_predictors_reject_bad_tta_before_any_engine():
    """The checks run before a checkpoint is read or an Engine created, so they need neither a file nor a GPU."""
    from bio_image_unet_b200 import multi_output_unet, multi_output_unet3d, siam_unet, unet, unet3d
    img2d = np.zeros((1, 64, 64), np.uint8)
    cases = [
        lambda: unet.Predict(img2d, 'x.tif', 'missing.pt', resize_dim=(32, 64), tta='dihedral', show_progress=False, device='cuda:0'),
        lambda: unet.Predict(img2d, 'x.tif', 'missing.pt', resize_dim=(64, 64), tta='mirror', show_progress=False, device='cuda:0'),
        lambda: unet.Session('missing.pt', resize_dim=(32, 64), tta='dihedral'),
        lambda: siam_unet.Predict(img2d, 'x.tif', 'missing.pt', resize_dim=(32, 64), tta='dihedral', show_progress=False, device='cuda:0'),
        lambda: siam_unet.Session('missing.pt', resize_dim=(64, 64), tta=1),
        lambda: unet3d.Predict(np.zeros((8, 32, 32), np.uint8), 'x.tif', 'missing.pt', resize_dim=(8, 32, 32),
                               tta='dihedral', progress_bar=False, device='cuda:0'),
        lambda: unet3d.Session('missing.pt', (8, 32, 32), tta='dihedral'),
        lambda: multi_output_unet3d.Predict(np.zeros((8, 32, 32), np.uint8), 'missing.pt', tta='dihedral',
                                            show_progress=False, device='cuda:0'),
        lambda: multi_output_unet3d.Session('missing.pt', tta='all'),
        lambda: multi_output_unet.Predict(np.zeros((40, 64), np.uint8), 'missing.pt', max_patch_size=(32, 64),
                                          tta='dihedral', show_progress=False, device='cuda:0'),
    ]
    for make in cases:
        with pytest.raises(ValueError):
            make()


def test_tta_extra_bytes():
    assert P.tta_extra_bytes(None, 3, (64, 64)) == 0
    assert P.tta_extra_bytes('flips', 2, (64, 64)) == 8 * 2 * 4096 + 4096
    assert P.tta_extra_bytes('flips', 1, (8, 16, 16), in_bytes=4) == 8 * 2048 + 4 * 2048


def test_oracle_tta_equals_hand_written_composition():
    sd = opipe._to_sd(_tiny_unet_sd())
    rng = np.random.default_rng(3)
    imgs = rng.integers(0, 4000, (1, 32, 32)).astype(np.uint16)
    got = oracle_tta_unet(imgs, sd, range(8), (32, 32))
    norm = opipe.preprocess_stack(imgs.copy(), 'single', (0., 99.8), False)
    x = torch.from_numpy(norm.astype('float32')[:, None] / 255)       # one tile = the whole image
    def f(sd, a):
        return omodels.FORWARD_2D['Unet'](sd, a)[0]
    with torch.no_grad():
        outs = [f(sd, x),
                f(sd, x.flip(-1)).flip(-1),
                f(sd, x.flip(-2)).flip(-2),
                f(sd, x.flip(-1).flip(-2)).flip(-2).flip(-1),
                f(sd, x.transpose(-2, -1)).transpose(-2, -1),
                f(sd, x.flip(-1).transpose(-2, -1)).transpose(-2, -1).flip(-1),
                f(sd, x.flip(-2).transpose(-2, -1)).transpose(-2, -1).flip(-2),
                f(sd, x.flip(-1).flip(-2).transpose(-2, -1)).transpose(-2, -1).flip(-2).flip(-1)]
    acc = outs[0]
    for o in outs[1:]:
        acc = acc + o
    want = ((acc * 0.125).numpy() * 255).astype('uint8')
    assert np.array_equal(got.reshape(want.shape), want)
    assert got.shape[-2:] == (32, 32)


def _tiny_unet_sd():
    from bio_image_unet_b200.unet import Unet
    torch.manual_seed(1)
    return Unet(n_filter=4).eval().state_dict()
