"""Multi-output 2D prediction of images / movies on B200 (reference: multi_output_unet/predict.py:13-285)."""
import os
from typing import Union

import numpy as np
import torch

from .. import pipeline2d as P
from .. import tiff
from ..engine import Engine
from ..progress import ProgressNotifier
from ..utils import get_device
from .multi_output_nested_unet import MultiOutputNestedUNet
from .multi_output_unet import MultiOutputUnet


def grid(shape, max_patch_size, add_tile):
    """Patch size (rounded up to a multiple of 16), tile counts, the linspace starts used for stitching and the
    sliding-window starts the patches are really taken at (multi_output_unet/predict.py:153-184: windows every
    X_start[1] pixels — not always the linspace positions, and not always N_x of them)."""
    _, h, w = shape
    ph = ((min(h, max_patch_size[0]) + 15) // 16) * 16
    pw = ((min(w, max_patch_size[1]) + 15) // 16) * 16
    n_x = int(np.ceil(h / ph)) + add_tile
    n_y = int(np.ceil(w / pw)) + add_tile
    hp, wp = h + max(ph - h, 0), w + max(pw - w, 0)
    xs = np.linspace(0, hp - ph, n_x).astype('uint16')
    ys = np.linspace(0, wp - pw, n_y).astype('uint16')
    sx = int(xs[1]) if n_x > 1 else 1
    sy = int(ys[1]) if n_y > 1 else 1
    if sx < 1 or sy < 1:
        raise ValueError('slice step cannot be zero')            # what the reference's [::0] raises (:181)
    wx = np.arange(0, hp - ph + 1, sx)
    wy = np.arange(0, wp - pw + 1, sy)
    return (ph, pw), n_x, n_y, xs, ys, wx, wy


class Predict:
    """Prediction of movies and images with the multi-output 2D U-Net (constructor surface of
    multi_output_unet/predict.py:16-19). Results per head in ``self.result`` (float32, when result_path is None)
    or as ``<result_path>_<head>.tif``.

    network : MultiOutputNestedUNet (U-Net++, the reference's default), MultiOutputNestedUNet_3Levels or
        MultiOutputUnet — the class of this package or of the reference, or its name. With a checkpoint trained with
        ``deep_supervision`` the last supervision head ('<head>_4' / '<head>_3') is used, like the reference's
        ``train_mode=False`` (multi_output_unet/predict.py:90-94, multi_output_nested_unet.py:143-145).
    The reference runs the model in float16 on CUDA devices and stores the result patches as float16; here the
    network runs in `precision` ('tf32' default | 'fp16' | 'bf16' | 'fp32', see unet.Predict) and the patches go
    through the same float16 rounding before the margin-weighted stitch. precision='fp16' is the reference's own
    arithmetic for this predictor: fp16 weights and activations, fp32 accumulation (the reference's float16
    convolutions accumulate in fp32 as well). Integer stacks (uint8 / uint16) are normalised on the device.
    tta (engine-only): None (default) | 'flips' (4 forwards per patch) | 'dihedral' (square patches: 8) - the head
    outputs of the flipped / rotated patches are mapped back and averaged in fp32 on the device; the mean goes through
    the float16 rounding and the margin-weighted stitch like an ordinary patch. It takes one more float32 buffer of
    all result patches.
    """

    def __init__(self, imgs, model_params, result_path=None, network=MultiOutputNestedUNet, max_patch_size=(1024, 1024),
                 batch_size=1, normalization_mode='single', clip_threshold=(0., 99.98), add_tile=0,
                 compress_tif=False, show_progress=True, device: Union[torch.device, str] = 'auto',
                 progress_notifier: ProgressNotifier = ProgressNotifier.progress_notifier_tqdm(), *,
                 precision='tf32', workspace_gb=24.0, keep_intermediates=False, tta=None):
        self.device = get_device() if device == 'auto' else torch.device(device)
        if isinstance(imgs, str):
            imgs = tiff.imread(imgs)
        self.max_patch_size = max_patch_size
        self.batch_size = batch_size
        self.add_tile = add_tile
        self.normalization_mode = normalization_mode
        self.clip_threshold = clip_threshold
        self.result_path = result_path
        self.compress_tif = compress_tif
        self.show_progress = show_progress
        name = network if isinstance(network, str) else getattr(network, '__name__', str(network))
        kinds = {'MultiOutputUnet': ('mo2d', 0), 'MultiOutputNestedUNet': ('nested2d', 4),
                 'MultiOutputNestedUNet_3Levels': ('nested2d_3l', 3)}
        if name not in kinds:
            raise ValueError(f"unknown network '{name}'")
        kind, depth = kinds[name]
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'normalization_mode {normalization_mode} not valid!')

        self.imgs_shape = imgs.shape
        if len(self.imgs_shape) == 2:
            imgs = np.expand_dims(imgs, axis=0)
            self.imgs_shape = imgs.shape
        if imgs.dtype not in (np.uint8, np.uint16):
            raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 stacks on the device; got {imgs.dtype}')
        (self.patch_size, self.N_x, self.N_y, self.X_start, self.Y_start, self._wx, self._wy) = grid(
            self.imgs_shape, max_patch_size, add_tile)
        self.tta = P.tta_codes(tta, 2, self.patch_size)

        self.model_params = torch.load(model_params, map_location='cpu')
        heads = self.model_params['output_heads']
        self.target_keys = list(heads.keys())
        if self.model_params['in_channels'] != 1:
            raise RuntimeError('multi_output_unet.Predict feeds single-channel patches (multi_output_unet/predict.py:208-210)')
        # deep supervision: inference reads the last supervision head (multi_output_nested_unet.py:143-145)
        suffix = f'_{depth}' if depth and self.model_params.get('deep_supervision', False) else ''
        self.engine = Engine(kind, self.model_params['state_dict'], self.model_params['n_filter'], 1,
                             [(k + suffix, heads[k]['channels'], heads[k].get('activation')
                               if heads[k].get('activation') in ('sigmoid', 'tanh', 'relu') else None)
                              for k in self.target_keys], precision=precision, device=self.device)
        self.N_per_img = self.N_x * self.N_y
        self.N = self.N_per_img * self.imgs_shape[0]

        result = self.__run(imgs, workspace_gb, keep_intermediates, progress_notifier)
        self.engine.close()
        del self.engine, self.model_params

        if self.result_path is not None:
            for key in self.target_keys:
                target = self.result_path + key + '.tif' if os.path.exists(self.result_path) else \
                    self.result_path + '_' + key + '.tif'
                tiff.imwrite(target, result[key], compression='deflate' if self.compress_tif else None)
            self.result = None
        else:
            self.result = result
        torch.cuda.empty_cache()

    def __run(self, imgs, workspace_gb, keep, progress_notifier):
        t, h, w = self.imgs_shape
        ph, pw = self.patch_size
        dev = self.device
        q_lo, q_hi = self.clip_threshold
        head_total = self.engine.head_total
        # normalisation (multi_output_unet/predict.py:128-151): float32 LUT of (clip(v) - min) / max
        frames = P.to_device_stack(imgs, dev)
        hist = P.E.histogram(frames)
        if self.normalization_mode == 'single':
            lut, _ = P.E.norm_lut_f32(hist, hist, t, q_lo, q_hi, 2)
        else:
            total = P.E.hist_sum(hist)
            bounds = total if self.normalization_mode == 'all' else hist[0:1].contiguous()
            lut, _ = P.E.norm_lut_f32(bounds, total, 1, q_lo, q_hi, 2)
        norm = P.E.apply_lut_f32(frames.reshape(t, -1), lut).reshape(t, 1, h, w)
        del frames
        # split: every sliding window (reflect padding at the far end when the image is smaller than the patch)
        n_win = len(self._wx) * len(self._wy)
        tile_batch = P.pick_tile_batch(self.engine, (ph, pw), t * n_win, int(workspace_gb * 2 ** 30))
        progress = progress_notifier.iterator if (self.tta is None and self.show_progress and
                                                  progress_notifier is not None) else None
        # (P, head_total, ph, pw) float32; with tta the mean over the transforms of every patch, stitched like a patch
        vals, patches = P.predict_tiles(
            lambda k: P.E.gather_tiles_f32_tta(norm, [0], self._wx, self._wy, (1, ph, pw), 2, k).reshape(-1, 1, ph, pw),
            lambda tl, on_val: P.run_tiles(self.engine, tl, tile_batch, want_val=True, want_u8=False, on_val=on_val,
                                           progress=progress),
            t * n_win, self.tta, 2, out_dtype=torch.float32)
        # stitch per head (the hole value is the mean of that head's float16 patches, :279)
        idx = (np.arange(t)[:, None, None] * self.N_per_img + np.arange(self.N_x)[None, :, None] * self.N_y +
               np.arange(self.N_y)[None, None, :]).astype(np.int32)
        if idx.max() >= patches.shape[0]:
            raise ValueError(f'cannot reshape array of size {patches.shape[0]} into tiles ({t}, {self.N_x}, {self.N_y})')
        src_index = torch.from_numpy(idx).to(dev)
        hs, ws = max(ph, h), max(pw, w)
        result, c0 = {}, 0
        heads = self.model_params['output_heads']
        for key in self.target_keys:
            c = heads[key]['channels']
            tiles_k = vals[:, c0:c0 + c].contiguous()
            fill = tiles_k.to(torch.float16).float().mean().to(torch.float16).float().reshape(1)
            st = P.E.stitch_margin_f32(tiles_k, src_index, t, c, (hs, ws), self.X_start, self.Y_start, (ph, pw), fill, 20)
            result[key] = np.squeeze(st[:, :, :h, :w].cpu().numpy())
            c0 += c
        if keep:
            self.norm = norm.reshape(t, h, w).cpu().numpy()
            self.patches = patches.reshape(-1, ph, pw).cpu().numpy()
            self.result_patches = vals.cpu().numpy()
        return result
