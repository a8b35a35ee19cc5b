"""Multi-output 3D prediction of (N, D, H, W) stacks on B200 (reference: multi_output_unet3d/predict.py:13-307)."""
import os
from typing import Union

import numpy as np
import torch

from .. import pipeline2d as P
from .. import tiff
from .. import tiling
from ..dist import DistContext
from ..engine import Engine
from ..progress import ProgressNotifier
from ..utils import get_device
from .multi_output_unet3d import MultiOutputUnet3D


class Session:
    """Reusable multi-output 3D predictor (checkpoint folded / packed once, workspace resident).
    precision: 'tf32' | 'fp16' | 'bf16' | 'fp32' (see unet.Predict); tta: None | 'flips' (see Predict)."""

    def __init__(self, model_params, max_patch_size=(64, 256, 256), overlap_factor=0.1, normalization_mode='single',
                 clip_threshold=(0., 99.98), device='cuda:0', precision='tf32', workspace_gb=24.0, dist=None, tta=None):
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'Invalid normalization mode: {normalization_mode}')
        self.tta = P.tta_codes(tta, 3, max_patch_size)
        params = torch.load(model_params, map_location='cpu') if isinstance(model_params, str) else model_params
        self.device = torch.device(device)
        self.max_patch_size, self.overlap_factor = max_patch_size, overlap_factor
        self.normalization_mode, self.clip_threshold = normalization_mode, clip_threshold
        self.workspace_bytes = int(workspace_gb * 2 ** 30)
        self.dist = dist if dist is not None else DistContext(False)
        self.output_heads = params['output_heads']
        self.target_keys = list(self.output_heads.keys())
        self.engine = Engine('mo3d', params['state_dict'], params['n_filter'], params['in_channels'],
                             [(k, self.output_heads[k]['channels'], self.output_heads[k].get('activation'))
                              for k in self.target_keys],
                             use_interpolation=params.get('use_interpolation', True), precision=precision,
                             device=self.device)
        self.tile_batch = None
        head_total = sum(self.output_heads[k]['channels'] for k in self.target_keys)
        self._planner = P.BatchPlanner(self.engine, self.workspace_bytes,
                                       lambda tile: P.tta_extra_bytes(tta, head_total, tile, in_bytes=4))
        self._pin = P.PinnedPool()
        self._host_out, self._s_out = None, None

    def _plan(self, tile, n_tiles):
        self.tile_batch = self._planner.ensure(tile, n_tiles)
        return self.tile_batch

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None

    def _normalise(self, vols_dev, lo):
        """float32 normalised copy of this rank's volumes (multi_output_unet3d/predict.py:104-125)."""
        q_lo, q_hi = self.clip_threshold
        n = vols_dev.shape[0]
        hist = P.E.histogram(vols_dev.reshape(n, -1)) if n else torch.zeros((0, P.E.HIST_BINS), dtype=torch.int32,
                                                                             device=self.device)
        if self.normalization_mode == 'single':
            lut, _ = P.E.norm_lut_f32(hist, hist, n, q_lo, q_hi, 0)
        else:
            part = P.E.hist_sum(hist) if n else torch.zeros((1, P.E.HIST_BINS), dtype=torch.int32, device=self.device)
            if self.normalization_mode == 'all':
                bounds = self.dist.all_reduce_sum(part)
            else:   # 'first': the statistics of volume 0, owned by rank 0
                bounds = hist[0:1].clone() if (lo == 0 and n) else torch.zeros((1, P.E.HIST_BINS), dtype=torch.int32,
                                                                               device=self.device)
                bounds = self.dist.all_reduce_sum(bounds)
            lut, _ = P.E.norm_lut_f32(bounds, bounds, 1, q_lo, q_hi, 1)
        return P.E.apply_lut_f32(vols_dev.reshape(n, -1), lut).reshape(vols_dev.shape) if n else \
            torch.zeros(vols_dev.shape, dtype=torch.float32, device=self.device)

    def predict(self, imgs, keep=False, progress_notifier=None, show_progress=False, to_host=True):
        """imgs: (N, D, H, W) (or (D, H, W)) uint8 / uint16 host stack -> {head: float32 array} on rank 0 (None
        elsewhere). Results are views of a pinned buffer that the next call reuses."""
        if imgs.ndim == 3:
            imgs = imgs[None]
        elif imgs.ndim != 4:
            raise ValueError(f'Unsupported input shape: {imgs.shape}')
        self.imgs_shape = tuple(imgs.shape)
        n_vol, d_img, h_img, w_img = imgs.shape
        self.patch_size = tuple(min(a, b) for a, b in zip((d_img, h_img, w_img), self.max_patch_size))
        self.Z_start = tiling.strided_starts(d_img, self.patch_size[0], self.overlap_factor)
        self.Y_start = tiling.strided_starts(h_img, self.patch_size[1], self.overlap_factor)
        self.X_start = tiling.strided_starts(w_img, self.patch_size[2], self.overlap_factor)
        self.N_z, self.N_y, self.N_x = len(self.Z_start), len(self.Y_start), len(self.X_start)
        self.N_per_vol = self.N_z * self.N_y * self.N_x
        lo, hi = self.dist.shard(n_vol)
        dev = self.device
        head_total = self.engine.head_total
        if imgs.dtype not in (np.uint8, np.uint16, torch.uint8, torch.uint16):
            raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 stacks on the device; got {imgs.dtype}')
        vols = P.to_device_stack(imgs[lo:hi].reshape(hi - lo, d_img * h_img, w_img), dev).reshape(hi - lo, d_img, h_img, w_img)
        norm = self._normalise(vols, lo)
        # multi-GPU: the stitched float32 volumes stay in HBM until the NCCL gather on rank 0
        on_device = self.dist.multi or not to_host
        shape = (hi - lo, head_total, d_img, h_img, w_img)
        if on_device:
            out_local = torch.zeros(shape, dtype=torch.float32, device=dev)
        else:
            # single process: chunks are copied back on a side stream into one (pinned, if it is not huge) host buffer
            # while the next chunk computes
            if self._host_out is None or tuple(self._host_out.shape) != shape:
                nbytes = 4 * int(np.prod(shape))
                self._host_out = torch.zeros(shape, dtype=torch.float32, pin_memory=nbytes <= (8 << 30))
            out_local = self._host_out
            if self._s_out is None:
                self._s_out = torch.cuda.Stream(dev)
            self._s_out.wait_stream(torch.cuda.current_stream(dev))
        if hi > lo:
            vols_per_chunk = max(1, min(hi - lo, self._planner.budget(self.patch_size) // self.N_per_vol))
            if hi - lo > 1:          # at least four chunks, so that the D2H copy of a chunk's result overlaps the next one
                vols_per_chunk = min(vols_per_chunk, max(1, -(-(hi - lo) // 4)))
            tile_batch = self._plan(self.patch_size, vols_per_chunk * self.N_per_vol)
            it = range(0, hi - lo, vols_per_chunk)
            if show_progress and self.dist.rank == 0 and progress_notifier is not None:
                it = progress_notifier.iterator(it)
            kept_p, kept_r = [], []
            for s in it:
                e = min(s + vols_per_chunk, hi - lo)
                # (n, head_total, pd, ph, pw); with tta the mean over the 8 flips, merged before the ramp blend
                vals, patches = P.predict_tiles(
                    lambda t: P.E.gather_tiles_f32_tta(norm[s:e], self.Z_start, self.Y_start, self.X_start,
                                                       self.patch_size, 3, t).reshape(-1, 1, *self.patch_size),
                    lambda tl, on_val: P.run_tiles(self.engine, tl, tile_batch, want_val=True, want_u8=False,
                                                   on_val=on_val),
                    (e - s) * self.N_per_vol, self.tta, 3, out_dtype=torch.float32)
                st = P.E.stitch_ramp_f32(vals, e - s, head_total, (d_img, h_img, w_img), self.Z_start, self.Y_start,
                                         self.X_start, self.patch_size, 16)
                if on_device:
                    out_local[s:e].copy_(st)
                else:
                    ev = torch.cuda.Event()
                    ev.record(torch.cuda.current_stream(dev))
                    with torch.cuda.stream(self._s_out):
                        self._s_out.wait_event(ev)
                        out_local[s:e].copy_(st, non_blocking=True)
                        st.record_stream(self._s_out)
                if keep:
                    kept_p.append(patches.cpu().numpy())
                    kept_r.append(vals.cpu().numpy())
            if keep:
                self.patches = np.concatenate(kept_p)
                self.result_patches = np.concatenate(kept_r)
        if on_device:
            full = self.dist.gather_slabs(out_local, self.dist.shards(n_vol))
            if not to_host:
                return full                  # (N, head_total, D, H, W) float32 device tensor (rank 0)
            full = None if full is None else self._pin.fetch('out', full)
        else:
            if self._s_out is not None:
                self._s_out.synchronize()
            full = out_local.numpy()
        if full is None:
            return None
        result, c0 = {}, 0
        heads = self.output_heads
        for key in self.target_keys:
            c = heads[key]['channels']
            result[key] = np.squeeze(full[:, c0:c0 + c])
            c0 += c
        return result


class Predict:
    """Prediction of volumetric (3D) data with the multi-output 3D U-Net (constructor surface of
    multi_output_unet3d/predict.py:16-27). Results per head in ``self.result`` (when result_path is None) or as
    ``<result_path>_<head>.tif``.

    normalization_mode='single' follows the reference's formula; the reference itself fails there on numpy >= 2
    (``ndarray.ptp`` was removed, :111). Integer stacks (uint8 / uint16) are normalised on the device.
    Engine-only keyword arguments: precision ('tf32' | 'fp16' | 'bf16' | 'fp32', see unet.Predict), workspace_gb,
    distributed (volumes are sharded over ranks), tta: None (default) or 'flips' - every patch also runs flipped along
    every combination of z, y and x (8 forwards per patch); the head outputs are flipped back and averaged in fp32 on
    the device before the ramp blend. About 8x the time of a plain prediction; memory stays within `workspace_gb`.
    """

    def __init__(self, imgs, model_params, result_path=None, network=MultiOutputUnet3D,
                 max_patch_size=(64, 256, 256), overlap_factor=0.1, batch_size=1, normalization_mode='single',
                 clip_threshold=(0., 99.98), add_tile=0, compress_tif=False, show_progress=True,
                 device: Union[torch.device, str] = 'auto',
                 progress_notifier: ProgressNotifier = ProgressNotifier.progress_notifier_tqdm(), *,
                 precision='tf32', workspace_gb=24.0, distributed=False, keep_intermediates=False, tta=None):
        P.tta_codes(tta, 3, max_patch_size)
        self.dist = DistContext(distributed)
        if device == 'auto':
            self.device = self.dist.device() if self.dist.active else get_device()
        else:
            self.device = torch.device(device)
        if isinstance(imgs, str):
            imgs = tiff.imread(imgs)
        self.max_patch_size = max_patch_size
        self.overlap_factor = overlap_factor
        self.batch_size = batch_size
        self.add_tile = add_tile
        self.normalization_mode = normalization_mode
        self.clip_threshold = clip_threshold
        self.result_path = result_path
        self.compress_tif = compress_tif
        self.show_progress = show_progress
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'Invalid normalization mode: {normalization_mode}')

        if imgs.ndim == 3:
            imgs = np.expand_dims(imgs, axis=0)
        elif imgs.ndim != 4:
            raise ValueError(f'Unsupported input shape: {imgs.shape}')
        self.imgs_shape = imgs.shape

        self.model_params = torch.load(model_params, map_location='cpu')
        ses = Session(self.model_params, max_patch_size, overlap_factor, normalization_mode, clip_threshold,
                      self.device, precision, workspace_gb, self.dist, tta=tta)
        self.target_keys = ses.target_keys
        result = ses.predict(imgs, keep=keep_intermediates, progress_notifier=progress_notifier,
                             show_progress=show_progress)
        for k in ('patch_size', 'Z_start', 'Y_start', 'X_start', 'N_z', 'N_y', 'N_x', 'N_per_vol'):
            setattr(self, k, getattr(ses, k))
        if keep_intermediates and hasattr(ses, 'patches'):
            self.patches, self.result_patches = ses.patches, ses.result_patches
        if result is not None:           # the session's pinned result buffer dies with it
            result = {k: np.array(v) for k, v in result.items()}
        self.fallback_ops = ses.engine.fallback_ops
        ses.close()
        del ses, self.model_params

        if result is None:
            self.result = None
        elif self.result_path is not None:
            for key in self.target_keys:
                target = self.result_path + key + '.tif' if os.path.exists(self.result_path) else \
                    self.result_path + '_' + key + '.tif'
                tiff.imwrite(target, result[key], compression='deflate' if self.compress_tif else None)
            self.result = None
        else:
            self.result = result
        torch.cuda.empty_cache()
