"""Tiled 2D U-Net prediction on B200 (reference: unet/predict.py:14-229; same constructor surface)."""
from typing import Union

import numpy as np
import torch

from .. import pipeline2d as P
from .. import tiff
from ..dist import DistContext
from ..engine import Engine
from ..progress import ProgressNotifier
from ..utils import get_device, save_as_tif
from .unet import Unet


class Session:
    """Reusable 2D predictor: checkpoint folded/packed once, weights and workspace resident on the device.

    ``predict(frames)`` takes a host (F, H, W) uint8/uint16 stack (ideally pinned) and returns the stitched
    (F, C, H, W) uint8 result on the host; ``predict_device`` does the same for a stack already in HBM.
    ``Predict`` (the reference's constructor-runs-everything class) is a thin wrapper around this.
    precision: 'tf32' | 'fp16' | 'bf16' | 'fp32', tta: None | 'flips' | 'dihedral', blend: None | 'gaussian' (see
    Predict).
    """

    KINDS = {'Unet': 'unet2d', 'AttentionUnet': 'attunet2d', 'Unet_v0': 'unet2d_v0'}

    def __init__(self, model_params, resize_dim=(512, 512), invert=False, normalization_mode='single',
                 clip_threshold=(0., 99.8), add_tile=0, device='cuda:0', precision='tf32', workspace_gb=24.0,
                 network='Unet', tta=None, blend=None):
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'normalization_mode {normalization_mode} not valid!')
        self.tta = P.tta_codes(tta, 2, resize_dim)
        self.blend = P.blend_mode(blend)
        params = torch.load(model_params, map_location='cpu') if isinstance(model_params, str) else model_params
        self.device = torch.device(device)
        self.resize_dim, self.add_tile, self.invert = tuple(resize_dim), add_tile, invert
        self.normalization_mode, self.clip_threshold = normalization_mode, clip_threshold
        self.out_channels = params['out_channels']
        self.workspace_bytes = int(workspace_gb * 2 ** 30)
        if network not in self.KINDS:
            raise ValueError(f"unknown network '{network}'")
        self.engine = Engine(self.KINDS[network], params['state_dict'], params['n_filter'], params['in_channels'],
                             [('', self.out_channels, 'sigmoid')], precision=precision, device=self.device)
        self.tile_batch = None
        self._planner = P.BatchPlanner(self.engine, self.workspace_bytes,
                                       lambda tile: P.tta_extra_bytes(tta, self.out_channels, tile))
        self.fixed_lut = None          # set by Predict for 'first' / 'all' (stack-wide statistics incl. other ranks)
        self.last = {}
        self._pin, self._streams, self._dev_in = P.PinnedPool(), None, None
        self._comm_stream, self._d2h_stream, self._slab, self._full, self.comm = None, None, None, None, {}

    def _ensure_plan(self, total_tiles):
        """Tile batch of the engine plan (pipeline2d.BatchPlanner: grows on demand, even split of the job over the
        forwards, no re-plan for the tail chunk of a movie)."""
        self.tile_batch = self._planner.ensure(self.resize_dim, total_tiles)

    def stack_lut(self, frames, chunk_frames, reduce=None, first_frame=None):
        """LUT of the 'first' / 'all' modes for a WHOLE integer stack (host or device, any length): bounds from frame 0
        / the whole stack, min / max from the whole stack (unet/predict.py:132-147). The stack is histogrammed chunk
        by chunk; `reduce` sums the totals over ranks; `first_frame` is frame 0 of the global stack when this rank's
        `frames` do not start there. Per-bin totals are kept in 64 bits and must fit the kernels' 32-bit counters."""
        dev = self.device
        total = torch.zeros((1, P.E.HIST_BINS), dtype=torch.int64, device=dev)
        for s0 in range(0, len(frames), max(1, chunk_frames)):
            chunk = frames[s0:s0 + chunk_frames]
            chunk = chunk.to(dev) if torch.is_tensor(chunk) else P.to_device_stack(chunk, dev)
            total += P.E.hist_sum(P.E.histogram(chunk.contiguous())).to(torch.int64) & 0xffffffff
        if reduce is not None:
            total = reduce(total)
        if int(total.max().item()) >= 2 ** 32:
            raise OverflowError('a single intensity value occurs in more than 2**32 pixels of the stack: the stack-wide '
                                "histogram of normalization_mode 'first' / 'all' does not fit its 32-bit counters")
        total = total.to(torch.int32)
        if self.normalization_mode == 'all':
            bounds = total
        else:
            f0 = frames[0:1] if first_frame is None else first_frame
            f0 = f0.to(dev) if torch.is_tensor(f0) else P.to_device_stack(f0, dev)
            bounds = P.E.histogram(f0.contiguous())
        lut, _ = P.E.norm_lut(bounds, total, 1, self.clip_threshold[0], self.clip_threshold[1], self.invert)
        return lut

    def lut_device(self, frames_dev, lut=None):
        """uint8 normalisation tables of an integer device stack: (F, 65536) in 'single' mode (per-frame statistics,
        unet/predict.py:123-131), (1, 65536) otherwise."""
        lut = lut if lut is not None else self.fixed_lut
        if lut is None and self.normalization_mode != 'single':     # the stack given here IS the whole stack
            lut = self.stack_lut(frames_dev, max(1, frames_dev.shape[0]))
        if lut is None:
            hist = P.E.histogram(frames_dev)
            lut, _ = P.E.norm_lut(hist, hist, frames_dev.shape[0], self.clip_threshold[0], self.clip_threshold[1],
                                  self.invert)
        return lut

    def normalise_device(self, frames_dev, lut=None):
        if frames_dev.dtype == torch.float32:
            # float stacks: exact float32 percentiles by radix select; 'first' / 'all' need the whole stack in one call
            u8, f32, _ = P.E.normalize_f32(frames_dev.contiguous(), self.normalization_mode, self.clip_threshold[0],
                                           self.clip_threshold[1], self.invert, want_f32=True)
            self.last_norm_f32 = f32
            return u8
        return P.E.apply_lut(frames_dev, self.lut_device(frames_dev, lut))

    def predict_device(self, frames_dev, keep=False, lut=None, planned=False, want_norm=None):
        """(F, H, W) uint8/uint16/float32 device tensor -> (F, C, H, W) uint8 device tensor. `lut`: stack-wide LUT when
        the frames are one chunk of a longer stack ('first' / 'all'); `planned`: the caller already sized the plan.
        Unless the normalised frames are wanted (`want_norm`, default = keep) the normalisation of an integer stack
        is fused into the tile gather and the normalised stack is never materialised."""
        f, h, w = frames_dev.shape
        if not planned:
            n_x, n_y, _, _ = P.tiling.grid_2d(h, w, self.resize_dim, self.add_tile)
            self._ensure_plan(f * n_x * n_y)
        want_norm = keep if want_norm is None else want_norm
        if frames_dev.dtype == torch.float32 or want_norm:
            src = norm = self.normalise_device(frames_dev, lut)
            lut = None
            if frames_dev.dtype == torch.float32:      # what the reference stores back into a float stack (:131)
                norm = self.last_norm_f32
        else:
            norm, src, lut = None, frames_dev.contiguous(), self.lut_device(frames_dev, lut)
        out, grid, tiles, res_tiles = P.predict_frames_2d(self.engine, src, self.resize_dim, self.add_tile,
                                                          self.out_channels, self.tile_batch, lut=lut, tta=self.tta,
                                                          blend=self.blend)
        self.last = dict(grid=grid, norm=norm, tiles=tiles if keep else None, result_tiles=res_tiles if keep else None)
        return out

    def predict(self, frames):
        """Host stack in, host result out (H2D and D2H inside, pipelined against the compute)."""
        return self.predict_movie(frames)[0]

    def predict_movie(self, frames, chunk_frames=None, want_norm=False, out_dev=None):
        """Pipelined prediction of a host (F, H, W) uint8/uint16 stack (numpy array or torch tensor, ideally
        pinned): the frames go through the device in chunks, and the H2D copy of chunk i+1 and the D2H copy of
        chunk i-1 run on their own streams while chunk i computes. Returns (result (F, C, H, W) uint8 numpy
        array backed by a pinned buffer that the next call reuses, normalised frames (F, H, W) uint8 or None).
        With `out_dev` (a (F, C, H, W) uint8 device tensor) the stitched frames stay on the device (multi-GPU runs
        gather them over NVLink before the one D2H copy on rank 0) and the first return value is `out_dev`."""
        if isinstance(frames, np.ndarray):
            if frames.dtype not in (np.uint8, np.uint16, np.float32):
                raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 / float32 stacks on the device; got '
                                f'{frames.dtype}. Convert the stack (e.g. to uint16 or float32) before calling Predict.')
            host = torch.from_numpy(np.ascontiguousarray(frames))
        else:
            if frames.dtype not in (torch.uint8, torch.uint16, torch.float32):
                raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 / float32 stacks on the device; got {frames.dtype}')
            host = frames.contiguous()
        resident = host.is_cuda             # the stack already lives in HBM: no H2D stage
        f, h, w = host.shape
        n_x, n_y, _, _ = P.tiling.grid_2d(h, w, self.resize_dim, self.add_tile)
        is_float = host.dtype == torch.float32
        if chunk_frames is None:
            self._ensure_plan(f * n_x * n_y)
            chunk_frames = max(1, min(f, self.tile_batch // (n_x * n_y)))
        if is_float and self.normalization_mode != 'single':
            chunk_frames = f               # stack-wide float statistics are taken in one pass over the whole stack
        self._ensure_plan(min(f, chunk_frames) * n_x * n_y)      # one chunk = a whole number of equal forwards
        dev = self.device
        lut = self.fixed_lut
        if lut is None and not is_float and self.normalization_mode != 'single' and f > chunk_frames:
            with torch.cuda.device(dev):   # stack-wide statistics first: the chunks must not use their own
                lut = self.stack_lut(host, chunk_frames)
        with torch.cuda.device(dev):
            if self._streams is None:
                self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev))
            s_in, s_comp, s_out = self._streams
            cur = torch.cuda.current_stream(dev)
            for st in self._streams:
                st.wait_stream(cur)
            out_host = self._pin.view('out', (f, self.out_channels, h, w), torch.uint8) if out_dev is None else None
            norm_host = self._pin.view('norm', (f, h, w), torch.float32 if is_float else torch.uint8) if want_norm else None
            pinned_in = resident or host.is_pinned()
            key = (chunk_frames, h, w, host.dtype)
            if not resident and (self._dev_in is None or self._dev_in[0] != key):
                self._dev_in = (key, [torch.empty((chunk_frames, h, w), dtype=host.dtype, device=dev) for _ in range(2)])
            dev_in = None if resident else self._dev_in[1]
            stage = None if pinned_in else [self._pin.view(f'stage{b}', (chunk_frames, h, w), host.dtype) for b in range(2)]
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_done = [torch.cuda.Event() for _ in range(2)]
            for i, s0 in enumerate(range(0, f, chunk_frames)):
                b = i & 1
                n = min(chunk_frames, f - s0)
                src = host[s0:s0 + n]
                if not pinned_in:
                    ev_in[b].synchronize()                      # the copy that last read this staging buffer is done
                    stage[b][:n].copy_(src)
                    src = stage[b][:n]
                if not resident:
                    with torch.cuda.stream(s_in):
                        s_in.wait_event(ev_done[b])             # the compute that last read dev_in[b] is done
                        dev_in[b][:n].copy_(src, non_blocking=True)
                        ev_in[b].record(s_in)
                with torch.cuda.stream(s_comp):
                    if not resident:
                        s_comp.wait_event(ev_in[b])
                    res = self.predict_device(src if resident else dev_in[b][:n], lut=lut, planned=True, want_norm=want_norm)
                    norm = self.last['norm'] if want_norm else None
                    if out_dev is not None:
                        out_dev[s0:s0 + n].copy_(res)
                    ev_done[b].record(s_comp)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_done[b])
                    if out_dev is None:
                        out_host[s0:s0 + n].copy_(res, non_blocking=True)
                        res.record_stream(s_out)
                    if want_norm:
                        norm_host[s0:s0 + n].copy_(norm, non_blocking=True)
                        norm.record_stream(s_out)
            s_out.synchronize()
            cur.wait_stream(s_comp)
        return (out_host.numpy() if out_dev is None else out_dev), (norm_host.numpy() if want_norm else None)

    def predict_movie_sharded(self, frames_local, ctx, n_total, chunk_frames=None, segments=4, to_host=True):
        """Multi-GPU prediction of a movie whose frames are sharded contiguously over the ranks of `ctx`
        (tiling.shard_range): `frames_local` is THIS rank's slice - a host stack (pinned ideally; H2D pipelined as in
        predict_movie) or a device tensor already in HBM. Frames are independent, so there is no data-path collective;
        the stitched uint8 slabs are gathered on rank 0 with NCCL send / recv over NVLink straight into a full-movie
        device buffer. The local slice is processed in `segments` parts: the gather of part j (communication stream)
        and, on rank 0, its D2H copy (copy stream) overlap the compute of part j + 1.

        Returns on rank 0 the (n_total, C, H, W) result - a numpy array backed by a pinned buffer (to_host) or the
        device tensor - and None elsewhere. ``self.comm`` holds {'bytes': received on rank 0, 'ms': NCCL time}."""
        dev = self.device
        f = int(frames_local.shape[0])
        lo, hi = ctx.shard(n_total)
        assert hi - lo == f, (lo, hi, f)
        h, w = int(frames_local.shape[1]), int(frames_local.shape[2])
        c = self.out_channels
        shards = ctx.shards(n_total)
        segments = max(1, min(segments, max(1, min(b - a for a, b in shards))))
        if self.normalization_mode != 'single' and self.fixed_lut is None:
            is_dev = torch.is_tensor(frames_local) and frames_local.is_cuda
            first = frames_local[0:1] if lo == 0 else None
            f0 = torch.zeros((1, h, w), dtype=torch.uint16, device=dev) if first is None else \
                (first if is_dev else P.to_device_stack(first, dev))
            if self.normalization_mode == 'first':      # frame 0 lives on rank 0
                f0 = ctx.broadcast(f0.view(torch.int16) if f0.dtype == torch.uint16 else f0, 0)
                f0 = f0.view(torch.uint16) if f0.dtype == torch.int16 else f0
            self.fixed_lut = self.stack_lut(frames_local, max(1, chunk_frames or 8), reduce=ctx.all_reduce_sum,
                                            first_frame=f0)
            clear_lut = True
        else:
            clear_lut = False
        with torch.cuda.device(dev):
            if self._comm_stream is None:
                self._comm_stream = torch.cuda.Stream(dev)
            s_comm = self._comm_stream
            if self._d2h_stream is None:
                self._d2h_stream = torch.cuda.Stream(dev)
            s_out = self._d2h_stream           # not predict_movie's copy stream: that one is synchronised per segment
            cur = torch.cuda.current_stream(dev)
            s_comm.wait_stream(cur)
            key = (f, c, h, w)
            if self._slab is None or self._slab[0] != key:
                self._slab = (key, torch.empty((f, c, h, w), dtype=torch.uint8, device=dev))
            slab = self._slab[1]
            full = None
            if ctx.rank == 0:
                if self._full is None or tuple(self._full.shape) != (n_total, c, h, w):
                    self._full = torch.empty((n_total, c, h, w), dtype=torch.uint8, device=dev) if ctx.multi else None
                full = self._full if ctx.multi else slab
            out_host = self._pin.view('out_full', (n_total, c, h, w), torch.uint8) if (to_host and ctx.rank == 0) else None
            t_ev = []
            for j in range(segments):
                a, b = P.tiling.shard_range(f, j, segments)
                if b > a:
                    self.predict_movie(frames_local[a:b], chunk_frames=chunk_frames, out_dev=slab[a:b])
                done = torch.cuda.Event()
                done.record(torch.cuda.current_stream(dev))
                bounds = []
                for r, (r_lo, r_hi) in enumerate(shards):
                    ra, rb = P.tiling.shard_range(r_hi - r_lo, j, segments)
                    bounds.append((r_lo + ra, r_lo + rb))
                with torch.cuda.stream(s_comm):
                    s_comm.wait_event(done)
                    if ctx.multi:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record(s_comm)
                        ctx.gather_slabs(slab[a:b], bounds, out=full, n_total=n_total)
                        e1.record(s_comm)
                        t_ev.append((e0, e1))
                    got = torch.cuda.Event()
                    got.record(s_comm)
                if out_host is not None:
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(got)
                        for ga, gb in bounds:
                            if gb > ga:
                                out_host[ga:gb].copy_(full[ga:gb], non_blocking=True)
            s_comm.synchronize()
            if out_host is not None:
                s_out.synchronize()
            cur.wait_stream(s_comm)
            self.comm = {'bytes': int((n_total - f) * c * h * w) if (ctx.multi and ctx.rank == 0) else 0,
                         'ms': float(sum(a.elapsed_time(b) for a, b in t_ev)) if t_ev else 0.0,
                         'collective': 'ncclSend/ncclRecv gather of the stitched uint8 slabs to rank 0 '
                                       f'({segments} segments, overlapped with compute)'}
        if clear_lut:
            self.fixed_lut = None
        if ctx.rank != 0:
            return None
        return out_host.numpy() if to_host else full

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
        self._pin.close()
        self._dev_in, self._slab, self._full = None, None, None


class Predict:
    """Prediction of movies and images with U-Net.

    1) load + intensity normalisation, 2) split into tiles of `resize_dim`, 3) U-Net forward, 4) stitch (mean of
    overlapping regions), 5) write a float16 TIFF — exactly the reference's steps, run as CUDA kernels.

    Parameters (identical to the reference, unet/predict.py:54-57)
    ----------
    imgs : ndarray or str      images to predict; a string is read as a TIFF file
    result_name : str          path of the result TIFF
    model_params : str         path of the checkpoint (.pt) written by the reference's Trainer
    network                    'Unet' | 'AttentionUnet' | 'Unet_v0' (string or class); None reads model_params['network']
    resize_dim                 tile size (multiples of 16)
    invert, normalization_mode ('single' | 'first' | 'all'), clip_threshold, add_tile, normalize_result,
    show_progress, device, progress_notifier : as in the reference

    Engine-only keyword arguments (defaults reproduce the reference's behaviour)
    ----------
    precision : 'tf32' (default, sigmoid within 1e-3 of the fp32 reference) | 'fp16' (tf32-grade error at the bf16
        speed; activations are stored as fp16, so values beyond +-65504 become +-inf as under the reference's
        model.half()) | 'bf16' (within 1e-2) | 'fp32'
    workspace_gb : activation workspace budget used to pick the tile batch size
    keep_intermediates : keep the uint8 tiles / result tiles as attributes (test hook)
    mutate_input : the reference overwrites the caller's array with the normalised frames in 'single' mode
        (unet/predict.py:131); kept by default
    distributed : shard frames over the ranks of an initialised torch.distributed process group (one GPU per rank)
    tta : test-time augmentation. None (default): one forward per tile. 'flips': the net also runs on the tiles
        flipped in x, in y and in both (4 forwards per tile); 'dihedral' (square `resize_dim` only): all 8 flips and
        rotations of the square (8 forwards). Each output is mapped back onto the tile, the float outputs are averaged
        in fp32 on the device, and the mean is quantised to uint8 once before the usual stitch. Costs about 4x / 8x
        the time of a plain prediction; tiles per forward and device memory stay within `workspace_gb`.
    blend : overlap stitch. None (default): the reference's mean of the overlapping tiles. 'gaussian': every tile's
        uint8 result is weighted by a centre-peaked Gaussian (sigma = tile / 8 per axis, tiling.gaussian_weights), so
        that pixels near a tile border, where the net saw the least context, count least; out = (sum w * v) // (sum w)
        in exact integer arithmetic. Composes with `tta` (the averaged tiles are blended).
    """

    def __init__(self, imgs, result_name, model_params, network='Unet', resize_dim=(512, 512),
                 invert=False, normalization_mode='single', clip_threshold=(0., 99.8), add_tile=0,
                 normalize_result=False, show_progress=True, device: Union[torch.device, str] = 'auto',
                 progress_notifier: ProgressNotifier = ProgressNotifier.progress_notifier_tqdm(), *,
                 precision='tf32', workspace_gb=24.0, mutate_input=True, distributed=False,
                 keep_intermediates=False, tta=None, blend=None):
        P.tta_codes(tta, 2, resize_dim)
        P.blend_mode(blend)
        self.dist = DistContext(distributed)
        self._keep = {'patches': [], 'result_patches': []} if keep_intermediates else None
        if device == 'auto':
            self.device = self.dist.device() if self.dist.active else get_device()
        else:
            self.device = torch.device(device)

        if isinstance(imgs, str):
            imgs = tiff.imread(imgs)

        self.resize_dim = resize_dim
        self.add_tile = add_tile
        self.normalize_result = normalize_result
        self.invert = invert
        self.normalization_mode = normalization_mode
        self.clip_threshold = clip_threshold
        self.result_name = result_name
        self.show_progress = show_progress
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'normalization_mode {normalization_mode} not valid!')

        imgs = self.__reshape_data(imgs)

        # checkpoint -> engine
        self.model_params = torch.load(model_params, map_location='cpu')
        if network is None:
            if 'network' in self.model_params.keys():
                network = self.model_params['network']
            else:
                raise ValueError('network is not defined')
        # strings as in unet/predict.py:89-97, or a class (the reference's or this package's) identified by name
        name = network if isinstance(network, str) else getattr(network, '__name__', str(network))
        if name not in Session.KINDS:
            raise ValueError(f"unknown network '{name}'")
        if name == 'Unet_v0' and 'in_channels' not in self.model_params.keys():
            self.model_params['in_channels'] = 1          # old checkpoints, unet/predict.py:95-97
            self.model_params['out_channels'] = 1
        out_channels = self.model_params['out_channels']
        if self.model_params['in_channels'] != 1:
            # the reference's tile array has a single channel (unet/predict.py:158) and its .view() fails otherwise
            raise RuntimeError("shape '[1, %d, %d, %d]' is invalid for input of size %d" % (
                self.model_params['in_channels'], resize_dim[0], resize_dim[1], resize_dim[0] * resize_dim[1]))
        self.session = Session(self.model_params, resize_dim, invert, normalization_mode, clip_threshold, add_tile,
                               self.device, precision, workspace_gb, network=name, tta=tta, blend=blend)

        # frames of this rank
        t_total = self.imgs_shape[0]
        lo, hi = self.dist.shard(t_total)
        self.N_x, self.N_y, self.X_start, self.Y_start = P.tiling.grid_2d(self.imgs_shape[1], self.imgs_shape[2],
                                                                          resize_dim, add_tile)
        self.N_per_img = self.N_x * self.N_y
        self.N = self.N_per_img * t_total
        print('Predicting data ...') if self.show_progress and self.dist.rank == 0 else None

        result_local = self.__run(imgs, lo, hi, out_channels, workspace_gb, mutate_input, progress_notifier)
        self.fallback_ops = self.session.engine.fallback_ops
        self.session.close()
        del self.session

        if self.dist.multi:
            # stitched uint8 slabs: NCCL send / recv over NVLink straight into rank 0's full-movie buffer, one D2H there
            full = self.dist.gather_slabs(result_local, self.dist.shards(t_total))
            imgs_result = None if full is None else full.cpu().numpy()
        else:
            imgs_result = result_local
        if imgs_result is not None:
            imgs_result = np.squeeze(imgs_result)
            save_as_tif(imgs_result, self.result_name, normalize=normalize_result)
        del self.model_params
        torch.cuda.empty_cache()

    def __reshape_data(self, imgs):
        self.imgs_shape = imgs.shape
        if len(self.imgs_shape) == 2:  # single image
            imgs = np.expand_dims(imgs, axis=0)
            self.imgs_shape = imgs.shape
        return imgs

    def __run(self, imgs, lo, hi, out_channels, workspace_gb, mutate_input, progress_notifier):
        th, tw = self.resize_dim
        h, w = self.imgs_shape[1:]
        n_local = hi - lo
        ses = self.session
        ses._ensure_plan(max(1, n_local * self.N_per_img))
        # frames per chunk: enough tiles to fill a few batches, bounded so the uint8 tile arrays stay small
        # (test-time augmentation keeps one fp32 sum per tile of a chunk: a chunk then holds at most one tile batch)
        chunk = max(1, min(max(n_local, 1), max(1, ((4 if ses.tta is None else 1) * ses.tile_batch) // self.N_per_img)))
        is_float = imgs.dtype == np.float32
        if is_float and self.normalization_mode in ('first', 'all'):
            if self.dist.active and self.dist.world > 1:
                raise NotImplementedError("float stacks with normalization_mode 'first' / 'all' are not sharded over ranks")
            chunk = max(n_local, 1)        # stack-wide float statistics: one pass over the whole stack on the device
        elif self.normalization_mode in ('first', 'all'):
            ses.fixed_lut = ses.stack_lut(imgs[lo:hi], chunk, reduce=self.dist.all_reduce_sum, first_frame=imgs[0:1])
        # multi-GPU: the stitched frames stay in HBM until the gather (a device tensor under NCCL; gloo gathers from the host)
        on_device = self.dist.multi and self._keep is None
        out = torch.zeros((n_local, out_channels, h, w), dtype=torch.uint8, device=self.device) if on_device else \
            np.zeros((n_local, out_channels, h, w), dtype='uint8')
        # super-chunks bound the pinned host buffers; inside one, copies and compute are pipelined
        frames_per_call = max(chunk, min(max(n_local, 1), (1 << 30) // max(h * w * max(out_channels, 2), 1)))
        starts = range(lo, hi, frames_per_call)
        it = progress_notifier.iterator(starts) if (self.show_progress and self.dist.rank == 0) else starts
        want_norm = self.normalization_mode == 'single' and mutate_input
        for s in it:
            e = min(s + frames_per_call, hi)
            if self._keep is not None:     # test hook: one chunk at a time, tiles copied out
                for c in range(s, e, chunk):
                    ce = min(c + chunk, e)
                    res = ses.predict_device(P.to_device_stack(imgs[c:ce], self.device), keep=True)
                    if want_norm:
                        imgs[c:ce] = ses.last['norm'].cpu().numpy()
                    out[c - lo:ce - lo] = res.cpu().numpy()
                    self._keep['patches'].append(ses.last['tiles'].cpu().numpy())
                    self._keep['result_patches'].append(ses.last['result_tiles'].cpu().numpy())
                continue
            res, norm = ses.predict_movie(imgs[s:e], chunk_frames=chunk, want_norm=want_norm,
                                          out_dev=out[s - lo:e - lo] if on_device else None)
            if want_norm:
                imgs[s:e] = norm                                # unet/predict.py:131 (cast back to the input dtype)
            if not on_device:
                out[s - lo:e - lo] = res
        if self._keep is not None:   # test hook: what the reference's __split / __predict return
            self.patches = np.concatenate(self._keep['patches'])
            self.result_patches = np.concatenate(self._keep['result_patches'])
        if self.dist.multi and not on_device:
            out = torch.from_numpy(out)
            out = out.to(self.device) if self.dist.backend == 'nccl' else out
        return out
