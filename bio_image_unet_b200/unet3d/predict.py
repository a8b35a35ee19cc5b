"""Patch-wise 3D U-Net prediction on B200 (reference: unet3d/predict.py:12-195)."""
from typing import Union

import numpy as np
import torch

from .. import pipeline2d as P
from .. import tiff
from .. import tiling
from ..dist import DistContext
from ..engine import Engine
from ..progress import ProgressNotifier
from ..utils import get_device, save_as_tif
from .unet3d import UNet3D


class Session:
    """Reusable 3D predictor: checkpoint folded / packed once; ``predict(vol)`` runs a (Z, X, Y) uint8 / uint16 host
    volume through normalise -> split -> forward -> mod-3 stitch and returns the uint8 result (on rank 0).
    precision: 'tf32' | 'fp16' | 'bf16' | 'fp32' (see unet.Predict); tta: None | 'flips', blend: None | 'gaussian'
    (see Predict)."""

    def __init__(self, model_params, resize_dim, invert=False, clip_threshold=(0., 99.8), add_patch=0, device='cuda:0',
                 precision='tf32', workspace_gb=24.0, dist=None, tta=None, blend=None):
        if len(resize_dim) != 3:
            raise IndexError('tuple index out of range')      # the reference indexes resize_dim[2] (:123)
        self.tta = P.tta_codes(tta, 3, resize_dim)
        self.blend = P.blend_mode(blend)
        params = torch.load(model_params, map_location='cpu') if isinstance(model_params, str) else model_params
        self.device = torch.device(device)
        self.resize_dim, self.invert, self.clip_threshold, self.add_patch = resize_dim, invert, clip_threshold, add_patch
        self.workspace_bytes = int(workspace_gb * 2 ** 30)
        self.out_channels = params['out_channels']
        self.dist = dist if dist is not None else DistContext(False)
        self.engine = Engine('unet3d', params['state_dict'], params['n_filter'], params['in_channels'],
                             [('', params['out_channels'], 'sigmoid')],
                             use_interpolation=params.get('use_interpolation', False), precision=precision,
                             device=self.device)
        self.tile_batch = None
        self._planner = P.BatchPlanner(self.engine, self.workspace_bytes,
                                       lambda tile: P.tta_extra_bytes(tta, params['out_channels'], tile))
        self.exchanged_bytes = 0
        self._pin = P.PinnedPool()
        self._s_out = None

    def _plan(self, tile, n_tiles):
        self.tile_batch = self._planner.ensure(tile, n_tiles)
        return self.tile_batch

    def _run_patches(self, src, lut, zs, patch):
        """uint8 result patches (n, 1, d, h, w) of the patch rows starting at `zs` of the (1, Z, X, Y) raw slab `src`
        (normalisation fused into the gather), and the plain uint8 patches; with test-time augmentation the result is
        the mean over the flips, merged on the device before the one uint8 quantisation."""
        n = len(zs) * len(self.X_start) * len(self.Y_start)
        tile_batch = self._plan(patch, n)
        res, patches = P.predict_tiles(
            lambda t: P.E.gather_tiles_tta(src, zs, self.X_start, self.Y_start, patch, 0, 3, t, lut=lut),
            lambda tl, on_val: P.run_tiles(self.engine, tl.reshape(n, 1, *patch), tile_batch, on_val=on_val),
            n, self.tta, 3)
        return patches, res

    def _stitch(self, tiles, n_planes, zs_local, patch):
        """Output planes [own_lo, own_lo + n_planes) from the uint8 result patches of consecutive z-rows whose starts,
        relative to own_lo, are zs_local (negative for rows that begin below): the reference's mod-3 rule, or the
        weighted stitch of blend='gaussian' (which does not depend on the patch order)."""
        x, y = self.vol_shape[1], self.vol_shape[2]
        if self.blend is None:
            return P.E.stitch_mod3_u8(tiles, (n_planes, x, y), zs_local, self.X_start, self.Y_start, patch)
        st = P.E.stitch_weighted_u8(tiles.contiguous(), 1, self.out_channels, (n_planes, x, y), zs_local, self.X_start,
                                    self.Y_start, patch, *P.blend_tables(patch))
        return st.view(n_planes, x, y)

    def _predict_pipelined(self, vol_dev, lut, zs, patch, shape, n_xy, groups=4):
        """Single process, host result wanted: the z-rows of the patch grid run in `groups` groups from the far end of
        the volume towards z = 0 (tiling.zslab_plan with the groups as virtual ranks: a group borrows only from groups
        that ran before it). Each group's output planes are stitched as soon as its patches are predicted and travel
        to the pinned host result on a copy stream while the next group computes."""
        d, h, w = patch
        z, x, y = shape
        dev = self.device
        plans = tiling.zslab_plan(zs, d, z, min(groups, self.N_z))
        out_host = self._pin.view('out', (z, x, y), torch.uint8)
        if self._s_out is None:
            self._s_out = torch.cuda.Stream(dev)
        cur = torch.cuda.current_stream(dev)
        self._s_out.wait_stream(cur)
        res_rows = {}
        src = vol_dev.contiguous().view(1, z, x, y)
        for g in reversed(range(len(plans))):
            lo, hi = plans[g]['rows']
            own_lo, own_hi = plans[g]['own']
            if hi <= lo:
                continue
            n = (hi - lo) * n_xy
            _, res = self._run_patches(src, lut, zs[lo:hi], (d, h, w))
            res = res.reshape(hi - lo, n_xy, d, h, w)
            for i, zi in enumerate(range(lo, hi)):
                res_rows[zi] = res[i]
            if own_hi > own_lo:
                extra = [zi for s in sorted(plans[g]['borrow']) for zi in plans[g]['borrow'][s]]
                st_rows = list(range(lo, hi)) + extra
                tiles = res.reshape(n, d, h, w) if not extra else torch.cat([res_rows[zi] for zi in st_rows])
                st = self._stitch(tiles, own_hi - own_lo, [zs[zi] - own_lo for zi in st_rows], (d, h, w))
                ev = torch.cuda.Event()
                ev.record(cur)
                with torch.cuda.stream(self._s_out):
                    self._s_out.wait_event(ev)
                    out_host[own_lo:own_hi].copy_(st, non_blocking=True)
                    st.record_stream(self._s_out)
        self._s_out.synchronize()
        return out_host.numpy()

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None

    def predict(self, vol, keep=False, to_host=True):
        """Single process: the whole volume. Multi-GPU: the z-rows of the patch grid (the outermost loop of
        unet3d/predict.py:146,180) are sharded contiguously; a rank uploads and normalises only the z-slab its rows
        touch, predicts its patches, receives from the ranks above it the uint8 result patches of the z-rows that
        reach down into its slab (their global patch index decides the mod-3 slot), stitches the output planes it
        owns, and the slabs are gathered on rank 0 - all device to device."""
        if vol.ndim == 2:
            vol = np.expand_dims(vol, axis=0)
        self.vol_shape = vol.shape
        (self.N_z, self.N_x, self.N_y, self.Z_start, self.X_start, self.Y_start) = tiling.grid_3d(
            self.vol_shape, self.resize_dim, self.add_patch)
        self.N = self.N_x * self.N_y * self.N_z
        d, h, w = (int(v) for v in self.resize_dim)
        z, x, y = self.vol_shape
        for starts, t, ext in ((self.Z_start, d, z), (self.X_start, h, x), (self.Y_start, w, y)):
            P.check_starts(starts, t, ext)
        dev = self.device
        ctx = self.dist
        zs = [int(v) for v in self.Z_start]
        n_xy = self.N_x * self.N_y
        plans = tiling.zslab_plan(zs, d, z, ctx.world)
        rows = [p['rows'] for p in plans]
        mine = plans[ctx.rank]
        (r_lo, r_hi), (a, b), (own_lo, own_hi) = mine['rows'], mine['slab'], mine['own']
        # global percentile normalisation: every rank histograms the planes it owns, one all-reduce, same LUT everywhere
        if b > a:
            slab_dev = P.to_device_stack(vol[a:b], dev)
            part = P.E.hist_sum(P.E.histogram(slab_dev[own_lo - a:own_hi - a].contiguous())) if own_hi > own_lo else None
        else:
            slab_dev, part = None, None
        if part is None:
            part = torch.zeros((1, P.E.HIST_BINS), dtype=torch.int32, device=dev)
        total = part.to(torch.int64) & 0xffffffff
        total = ctx.all_reduce_sum(total)
        if ctx.multi and int(total.max().item()) >= 2 ** 32:
            raise OverflowError('a single intensity value occurs in more than 2**32 voxels: the global histogram does '
                                'not fit its 32-bit counters')
        total = total.to(torch.int32)
        lut, _ = P.E.norm_lut(total, total, 1, self.clip_threshold[0], self.clip_threshold[1], self.invert)
        if not ctx.multi and to_host and not keep and self.N_z >= 2:
            return self._predict_pipelined(slab_dev, lut, zs, (d, h, w), (z, x, y), n_xy)
        n_local = (r_hi - r_lo) * n_xy
        if n_local > 0:
            # normalisation fused into the patch gather: the normalised (b - a, X, Y) slab is never written
            patches, res_local = self._run_patches(slab_dev.contiguous().view(1, b - a, x, y), lut,
                                                   [v - a for v in zs[r_lo:r_hi]], (d, h, w))
            del slab_dev
            res_local = res_local.reshape(n_local, d, h, w)
        else:
            patches = torch.zeros((0, d, h, w), dtype=torch.uint8, device=dev)
            res_local = torch.zeros((0, d, h, w), dtype=torch.uint8, device=dev)

        # rows of higher ranks that reach into a lower rank's slab travel down (NCCL send / recv of uint8 patches)
        sends, recvs, extra_rows = [], [], []
        if ctx.multi:
            for r in range(ctx.rank):
                need = plans[r]['borrow'].get(ctx.rank)
                if need:
                    i0, i1 = (need[0] - r_lo) * n_xy, (need[-1] + 1 - r_lo) * n_xy
                    sends.append((r, res_local[i0:i1]))
            for s in range(ctx.rank + 1, ctx.world):
                need = mine['borrow'].get(s)
                if need:
                    buf = torch.empty((len(need) * n_xy, d, h, w), dtype=torch.uint8, device=dev)
                    recvs.append((s, buf))
                    extra_rows += need
            ctx.exchange(sends, recvs)
            self.exchanged_bytes = sum(int(t.numel()) for _, t in sends) + sum(int(t.numel()) for _, t in recvs)
        # stitch the planes this rank owns from its own rows + the borrowed ones (consecutive rows r_lo .. r_lo + k - 1:
        # their local patch index is the global one minus r_lo * N_x * N_y, which only relabels the three slots)
        if own_hi > own_lo:
            assert extra_rows == list(range(r_hi, r_hi + len(extra_rows)))
            tiles = torch.cat([res_local] + [t for _, t in recvs]) if recvs else res_local
            st_rows = list(range(r_lo, r_hi + len(extra_rows)))
            st = self._stitch(tiles, own_hi - own_lo, [zs[zi] - own_lo for zi in st_rows], (d, h, w))
        else:
            st = torch.zeros((0, x, y), dtype=torch.uint8, device=dev)
        if keep:       # test hook: what the reference's __split / __predict return (gathered on rank 0)
            bounds_p = [(lo * n_xy, hi * n_xy) for lo, hi in rows]
            allp, allr = ctx.gather_slabs(patches.reshape(n_local, d, h, w), bounds_p), ctx.gather_slabs(res_local, bounds_p)
            if allp is not None:
                self.patches, self.result_patches = allp.cpu().numpy(), allr.cpu().numpy()
        full = ctx.gather_slabs(st, [p['own'] for p in plans], n_total=z) if ctx.multi else st
        if full is None or not to_host:
            return full
        return self._pin.fetch('out', full)      # view of a pinned buffer that the next call reuses


class Predict:
    """Prediction of movies or 3D stacks with 3D U-Net (constructor surface of unet3d/predict.py:52-55).

    `normalization_mode` is accepted and unused, as in the reference: percentiles are always taken over the whole
    volume (unet3d/predict.py:109-117). Engine-only keyword arguments as in unet.Predict (precision 'tf32' | 'fp16' |
    'bf16' | 'fp32'); with `distributed=True`
    the z-rows of the patch grid are sharded over ranks: each rank uploads only its z-slab, the intensity histogram
    is all-reduced, boundary patches are exchanged point to point, every rank stitches the planes it owns and rank
    0 gathers the uint8 slabs (all device to device).

    tta (engine-only): None (default) or 'flips': the net also runs on the patches flipped along every combination of
    z, y and x (8 forwards per patch); the outputs are flipped back, averaged in fp32 on the device and quantised to
    uint8 once before the mod-3 stitch. About 8x the time of a plain prediction; memory stays within `workspace_gb`.

    blend (engine-only): None (default, the reference's mod-3 stitch) or 'gaussian': the overlapping uint8 result
    patches are merged as (sum w * v) // (sum w) with w = w_d[tz] * w_h[ty] * w_w[tx], Gaussian tables with sigma =
    patch / 8 per axis (tiling.gaussian_weights), so that voxels near a patch border count least. Exact integer
    arithmetic: sharding and z-row groups do not change a byte. Composes with `tta`.
    """

    def __init__(self, vol, result_name, model_params, network=UNet3D, resize_dim=(512, 512),
                 invert=False, normalization_mode='single', clip_threshold=(0., 99.8), add_patch=0,
                 normalize_result=False, progress_bar=True, device: Union[torch.device, str] = 'auto',
                 progress_notifier: ProgressNotifier = ProgressNotifier.progress_notifier_tqdm(), *,
                 precision='tf32', workspace_gb=24.0, distributed=False, keep_intermediates=False, tta=None,
                 blend=None):
        if len(resize_dim) == 3:
            P.tta_codes(tta, 3, resize_dim)
        P.blend_mode(blend)
        if isinstance(vol, str):
            vol = tiff.imread(vol)
        self.dist = DistContext(distributed)
        if device == 'auto':
            self.device = self.dist.device() if self.dist.active else get_device()
        else:
            self.device = torch.device(device)
        self.resize_dim = resize_dim
        self.add_patch = add_patch
        self.normalize_result = normalize_result
        self.invert = invert
        self.normalization_mode = normalization_mode
        self.clip_threshold = clip_threshold
        self.result_name = result_name
        self.progress_bar = progress_bar

        self.vol_shape = vol.shape
        if len(self.vol_shape) == 2:
            vol = np.expand_dims(vol, axis=0)
            self.vol_shape = vol.shape

        self.model_params = torch.load(model_params, map_location='cpu')
        ses = Session(self.model_params, resize_dim, invert, clip_threshold, add_patch, self.device, precision,
                      workspace_gb, self.dist, tta=tta, blend=blend)
        print('Predicting data ...') if self.progress_bar and self.dist.rank == 0 else None
        vol_result = ses.predict(vol, keep=keep_intermediates)
        for k in ('N_z', 'N_x', 'N_y', 'Z_start', 'X_start', 'Y_start', 'N'):
            setattr(self, k, getattr(ses, k))
        if keep_intermediates and hasattr(ses, 'patches'):
            self.patches, self.result_patches = ses.patches, ses.result_patches
        self.fallback_ops = ses.engine.fallback_ops
        ses.close()
        del ses
        if vol_result is not None:
            save_as_tif(np.squeeze(vol_result), self.result_name, normalize=normalize_result)
        del self.model_params
        torch.cuda.empty_cache()
