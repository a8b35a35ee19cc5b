"""Tiled Siamese U-Net prediction of TIFF movies on B200 (reference: siam_unet/predict.py:15-240).

The reference walks the movie frame by frame: read page i (and i-1), pair = (previous, current) with frame 0 paired
with frame 1, normalise the pair, split both frames into tiles, forward each tile pair, stitch, append the page to
the TIFF writer. Here the movie STREAMS through the device in chunks of pairs: the pages of chunk i+1 are read from
the TIFF and copied to the device while chunk i computes and the stitched pages of chunk i-1 travel back and are
appended to the result TIFF (three CUDA streams, pinned double buffers) - neither the input movie nor the result is
ever held in host memory as a whole. In 'single' mode each frame is normalised once (its normalised form is the same
in both pairs it belongs to).
"""
import os
from typing import Union

import numpy as np
import torch

from .. import pipeline2d as P
from .. import tiff
from ..dist import DistContext
from ..engine import Engine
from ..progress import ProgressNotifier
from ..utils import get_device


def _take(frames, sel):
    """frames[sel] for uint8 / uint16 device stacks (torch has no CUDA index kernel for uint16)."""
    if frames.dtype == torch.uint16:
        return frames.view(torch.int16)[sel].contiguous().view(torch.uint16)
    return frames[sel].contiguous()


class _ArraySource:
    """(T, H, W) ndarray as a page source."""

    def __init__(self, movie):
        self.movie = movie[None] if movie.ndim == 2 else movie
        self.n, self.shape, self.dtype = self.movie.shape[0], tuple(self.movie.shape[1:]), self.movie.dtype

    def read_into(self, dst, indices):
        for k, i in enumerate(indices):
            dst[k] = self.movie[i]


class _TiffSource:
    """TIFF pages read on demand, one page at a time like siam_unet/predict.py:110-115."""

    def __init__(self, path):
        self.path = path
        self.n, self.shape = tiff.page_count_and_shape(path)
        self.dtype = tiff.imread(path, key=0).dtype

    def read_into(self, dst, indices):
        for k, i in enumerate(indices):
            dst[k] = tiff.imread(self.path, key=int(i))


class Session:
    """Reusable Siamese predictor: checkpoint folded / packed once, weights and workspace resident on the device.
    ``predict_stream`` runs pairs [lo, hi) of a page source through the three-stream pipeline.
    precision: 'tf32' | 'fp16' | 'bf16' | 'fp32', tta: None | 'flips' | 'dihedral' (see unet.Predict; both frames of
    a pair get the same transform), blend: None | 'gaussian' (see unet.Predict)."""

    def __init__(self, model_params, resize_dim=(512, 512), invert=False, normalization_mode='single',
                 clip_threshold=(0.0, 99.98), add_tile=0, device='cuda:0', precision='tf32', workspace_gb=24.0,
                 tta=None, blend=None):
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'normalization_mode {normalization_mode} not valid!')
        P.tta_codes(tta, 2, resize_dim if resize_dim is not None else (1, 1))   # whole frames: checked per frame size
        self.blend = P.blend_mode(blend)
        self.tta_mode = tta
        params = torch.load(model_params, map_location='cpu') if isinstance(model_params, str) else model_params
        self.device = torch.device(device)
        self.resize_dim, self.add_tile, self.invert = resize_dim, add_tile, invert
        self.normalization_mode, self.clip_threshold = normalization_mode, clip_threshold
        self.workspace_bytes = int(workspace_gb * 2 ** 30)
        self.engine = Engine('siam2d', params['state_dict'], params['n_filter'], 1, [('', 1, 'sigmoid')],
                             siam_mode=params['mode'], precision=precision, device=self.device)
        self.tile_batch = None
        self._planner = P.BatchPlanner(self.engine, self.workspace_bytes,
                                       lambda tile: P.tta_extra_bytes(tta, 1, tile, in_bytes=2))
        # per-frame normalisation + a join that uses the previous frame: frame t's encoder pass serves pair t (as the
        # current frame) and pair t + 1 (as the previous one) - it runs once (biu_net_set_siam_shared)
        self.shared_encoder = normalization_mode == 'single' and params['mode'] != 'control'
        self.siam_mode = params['mode']
        self._pin, self._streams, self._dev_in = P.PinnedPool(), None, None
        self.last = {}

    # ---- geometry / planning ---------------------------------------------------------------------------------
    def grid(self, h, w):
        rd = self.resize_dim if self.resize_dim is not None else (h, w)
        return (rd, *P.tiling.grid_2d(h, w, rd, self.add_tile))

    def _ensure_plan(self, rd, total_tiles, n_per=0):
        self._planner.plan_kwargs = {'siam_shared': n_per} if (self.shared_encoder and n_per) else {}
        self.tile_batch = self._planner.ensure(rd, total_tiles)

    def chunk_frames(self, n_frames, s, e):
        """Frames a chunk of pairs [s, e) needs, in upload order, and the (previous, current) position of every pair.
        Shared encoder: [previous frame of pair s, frames s .. e-1] - pair j is (position j, position j + 1)."""
        prev_idx, cur_idx = self.pair_indices(n_frames, s, e)
        if self.shared_encoder:
            needed = [prev_idx[0]] + cur_idx
            return needed, list(range(e - s)), list(range(1, e - s + 1))
        needed = sorted(set(prev_idx + cur_idx))
        pos = {f: j for j, f in enumerate(needed)}
        return needed, [pos[f] for f in prev_idx], [pos[f] for f in cur_idx]

    @staticmethod
    def pair_indices(n_frames, lo, hi):
        """(previous, current) frame index of every pair in [lo, hi) (siam_unet/predict.py:107-117)."""
        prev = [(1 if n_frames > 1 else 0) if i == 0 else i - 1 for i in range(lo, hi)]
        return prev, list(range(lo, hi))

    # ---- one chunk on the device -------------------------------------------------------------------------------
    def predict_pairs_device(self, frames, p_sel, c_sel, keep=False):
        """frames: (K, H, W) uint8/uint16 device stack holding every frame the pairs need; p_sel / c_sel: int64 device
        index tensors (previous / current frame of each pair). Returns the stitched (n_pairs, 1, H, W) uint8 tensor."""
        k, h, w = frames.shape
        rd, n_x, n_y, xs, ys = self.grid(h, w)
        th, tw = rd
        tta = P.tta_codes(self.tta_mode, 2, rd)
        n_pairs = int(c_sel.shape[0])
        q_lo, q_hi = self.clip_threshold
        hist = P.E.histogram(frames)
        if self.shared_encoder:
            # frames = [previous frame of the first pair | current frames] (chunk_frames): every frame is normalised on
            # its own statistics (:128-136) inside the tile gather, and its tiles go through the encoder once
            assert k == n_pairs + 1, 'shared encoder: the stack must hold the n_pairs + 1 frames of chunk_frames()'
            P.check_starts(xs, th, h)
            P.check_starts(ys, tw, w)
            lut, _ = P.E.norm_lut(hist, hist, k, q_lo, q_hi, self.invert)
            n_per = n_x * n_y
            src = frames.contiguous().view(k, 1, h, w)
            # with tta every unique tile of a pass carries the same transform: the shared encoder runs as it is
            res_u8, tiles_u = P.predict_tiles(
                lambda t: P.E.gather_tiles_tta(src, [0], xs, ys, (1, th, tw), 1, 2, t, lut=lut),
                lambda tl, on_val: P.run_tiles(self.engine, tl, self.tile_batch, n_per=n_per, on_val=on_val),
                n_pairs * n_per, tta, 2)
            st = P.stitch_2d(res_u8, n_pairs, 1, (h, w), xs, ys, (th, tw), self.blend)
            self.last = dict(tiles_cur=tiles_u[n_per:], tiles_prev=tiles_u[:n_pairs * n_per], result_tiles=res_u8) if keep else {}
            return st
        if self.normalization_mode == 'single':       # each frame on its own statistics (:128-136)
            lut, _ = P.E.norm_lut(hist, hist, k, q_lo, q_hi, self.invert)
            norm = P.E.apply_lut(frames, lut)
            norm_prev, norm_cur = norm[p_sel].contiguous(), norm[c_sel].contiguous()
        else:                                          # statistics of the pair (:137-152): stack = [prev, cur]
            pair_range = (hist[p_sel] + hist[c_sel]).contiguous()
            bounds = hist[p_sel].contiguous() if self.normalization_mode == 'first' else pair_range
            lut, _ = P.E.norm_lut(bounds, pair_range, n_pairs, q_lo, q_hi, self.invert)
            norm_prev = P.E.apply_lut(_take(frames, p_sel), lut)
            norm_cur = P.E.apply_lut(_take(frames, c_sel), lut)
        P.check_starts(xs, th, h)
        P.check_starts(ys, tw, w)
        # zero padding; with tta both frames of a pair get the same transform
        res_u8, (tiles_cur, tiles_prev) = P.predict_tiles(
            lambda t: tuple(P.E.gather_tiles_tta(nf.view(n_pairs, 1, h, w), [0], xs, ys, (1, th, tw), 1, 2, t)
                            for nf in (norm_cur, norm_prev)),
            lambda tl, on_val: P.run_tiles(self.engine, tl[0], self.tile_batch, prev_tiles=tl[1], on_val=on_val),
            n_pairs * n_x * n_y, tta, 2)
        st = P.stitch_2d(res_u8, n_pairs, 1, (h, w), xs, ys, (th, tw), self.blend)
        self.last = dict(tiles_cur=tiles_cur, tiles_prev=tiles_prev, result_tiles=res_u8) if keep else {}
        return st

    # ---- the streaming pipeline --------------------------------------------------------------------------------
    def predict_stream(self, source, lo, hi, sink, chunk_pairs=None, keep=None, progress=None, out_dev=None):
        """Pairs [lo, hi) of `source` (an object with n / shape / dtype / read_into(dst, frame_indices)) through the
        device; `sink(first_pair, frames_u8)` receives the stitched (n, H, W) uint8 pages of each chunk in order (a
        view of a pinned buffer, valid until the next-but-one chunk). With `out_dev` the pages stay on the device."""
        h, w = source.shape
        rd, n_x, n_y, xs, ys = self.grid(h, w)
        n_per = n_x * n_y
        if hi <= lo:
            return
        if chunk_pairs is None:
            self._ensure_plan(rd, (hi - lo) * n_per, n_per)
            chunk_pairs = max(1, min(hi - lo, max(1, self.tile_batch // n_per)))
        self._ensure_plan(rd, min(hi - lo, chunk_pairs) * n_per, n_per)
        tdtype = {np.dtype('uint8'): torch.uint8, np.dtype('uint16'): torch.uint16}.get(np.dtype(source.dtype))
        if tdtype is None:
            raise TypeError(f'bio_image_unet_b200 normalises uint8 / uint16 movies on the device; got {source.dtype}')
        dev = self.device
        kmax = chunk_pairs + 2
        with torch.cuda.device(dev):
            if self._streams is None:
                self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev))
            s_in, s_comp, s_out = self._streams
            cur = torch.cuda.current_stream(dev)
            for st in self._streams:
                st.wait_stream(cur)
            key = (kmax, h, w, tdtype)
            if self._dev_in is None or self._dev_in[0] != key:
                self._dev_in = (key, [torch.empty((kmax, h, w), dtype=tdtype, device=dev) for _ in range(2)])
            dev_in = self._dev_in[1]
            stage = [self._pin.view(f'stage{b}', (kmax, h, w), tdtype) for b in range(2)]
            outb = [self._pin.view(f'out{b}', (chunk_pairs, h, w), torch.uint8) for b in range(2)]
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_done = [torch.cuda.Event() for _ in range(2)]
            ev_out = [torch.cuda.Event() for _ in range(2)]
            pending = [None, None]                       # (first pair, count) whose D2H copy sits in outb[b]

            def flush(b):
                if pending[b] is not None:
                    ev_out[b].synchronize()
                    s0, n = pending[b]
                    sink(s0, outb[b][:n].numpy())
                    pending[b] = None

            starts = list(range(lo, hi, chunk_pairs))
            it = progress.iterator(starts) if progress is not None else starts
            for i, s in enumerate(it):
                b = i & 1
                e = min(s + chunk_pairs, hi)
                needed, p_pos, c_pos = self.chunk_frames(source.n, s, e)
                k = len(needed)
                ev_in[b].synchronize()                  # the H2D copy that last read this staging buffer is done
                source.read_into(stage[b].numpy(), needed)      # host work overlaps the previous chunk's kernels
                p_sel = P.E._dev_i64(p_pos, dev)
                c_sel = P.E._dev_i64(c_pos, dev)
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_done[b])         # the compute that last read dev_in[b] is done
                    dev_in[b][:k].copy_(stage[b][:k], non_blocking=True)
                    ev_in[b].record(s_in)
                flush(b)                                # outb[b] is about to be rewritten: hand its pages over first
                with torch.cuda.stream(s_comp):
                    s_comp.wait_event(ev_in[b])
                    st = self.predict_pairs_device(dev_in[b][:k], p_sel, c_sel, keep=keep is not None)
                    if out_dev is not None:
                        out_dev[s - lo:e - lo].copy_(st[:, 0])
                    ev_done[b].record(s_comp)
                    if keep is not None:              # test hook (on the compute stream: .cpu() waits for the kernels)
                        both = torch.stack((self.last['tiles_cur'][:, 0], self.last['tiles_prev'][:, 0]), dim=1)
                        keep['patches'].append(both.cpu().numpy().reshape(e - s, n_per, 2, *rd))
                        keep['result_patches'].append(self.last['result_tiles'].cpu().numpy().reshape(e - s, n_per, 1, *rd))
                if out_dev is None:
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(ev_done[b])
                        outb[b][:e - s].copy_(st[:, 0], non_blocking=True)
                        st.record_stream(s_out)
                        ev_out[b].record(s_out)
                    pending[b] = (s, e - s)
                flush(b ^ 1)                            # the previous chunk's pages: written while this chunk computes
            flush(0)
            flush(1)
            s_comp.synchronize()
            cur.wait_stream(s_comp)

    def close(self):
        if self.engine is not None:
            self.engine.close()
            self.engine = None
        self._pin.close()
        self._dev_in = None


class Predict:
    """Prediction of tif-movies with Siamese U-Net (constructor surface of siam_unet/predict.py:53-56).

    tif_file : str (an ndarray (T, H, W) is also accepted); resize_dim=None processes whole frames.
    Engine-only keyword arguments: precision ('tf32' | 'fp16' | 'bf16' | 'fp32'), workspace_gb, distributed,
    keep_intermediates, tta (None | 'flips' | 'dihedral'; see unet.Predict). With tta both frames of a pair get the
    same flip / rotation, and the shared-encoder mode stays shared. blend (None | 'gaussian'; see unet.Predict): with
    resize_dim=None every frame is one tile, so there is nothing to blend and the result is the same.
    """

    def __init__(self, tif_file, result_name, model_params, resize_dim=(512, 512), invert=False,
                 normalization_mode='single', clip_threshold=(0.0, 99.98), add_tile=0, normalize_result=False,
                 show_progress=True, device: Union[torch.device, str] = 'auto',
                 progress_notifier: ProgressNotifier = ProgressNotifier.progress_notifier_tqdm(), *,
                 precision='tf32', workspace_gb=24.0, distributed=False, keep_intermediates=False, tta=None,
                 blend=None):
        P.tta_codes(tta, 2, resize_dim if resize_dim is not None else (1, 1))
        P.blend_mode(blend)
        self.dist = DistContext(distributed)
        if device == 'auto':
            self.device = self.dist.device() if self.dist.active else get_device()
        else:
            self.device = torch.device(device)
        self.tif_file = tif_file
        self.add_tile = add_tile
        self.invert = invert
        self.normalization_mode = normalization_mode
        self.clip_threshold = clip_threshold
        self.result_name = result_name
        self.normalize_result = normalize_result
        self.show_progress = show_progress
        self.progress_notifier = progress_notifier
        if normalization_mode not in ('single', 'first', 'all'):
            raise ValueError(f'normalization_mode {normalization_mode} not valid!')

        # load model
        self.model_params = torch.load(model_params, map_location='cpu')
        self.session = Session(self.model_params, resize_dim, invert, normalization_mode, clip_threshold, add_tile,
                               self.device, precision, workspace_gb, tta=tta, blend=blend)

        if isinstance(tif_file, str):
            source = _TiffSource(tif_file)
            os.makedirs(f'temp_{tif_file.split("/")[-1]}', exist_ok=True)    # siam_unet/predict.py:88,100
        else:
            source = _ArraySource(np.asarray(tif_file))
        self.tif_len = source.n
        self.imgs_shape = [self.tif_len, source.shape[0], source.shape[1]]
        self.resize_dim = resize_dim if resize_dim is not None else (self.imgs_shape[1], self.imgs_shape[2])
        self.session.resize_dim = self.resize_dim

        self.N_x, self.N_y, self.X_start, self.Y_start = P.tiling.grid_2d(self.imgs_shape[1], self.imgs_shape[2],
                                                                          self.resize_dim, add_tile)
        self.N_per_img = self.N_x * self.N_y
        self.N = self.N_x * self.N_y
        self._keep = {'patches': [], 'result_patches': []} if keep_intermediates else None

        print('Predicting data ...') if self.show_progress and self.dist.rank == 0 else None
        lo, hi = self.dist.shard(self.tif_len)
        h, w = self.imgs_shape[1:]
        progress = self.progress_notifier if (self.show_progress and self.dist.rank == 0) else None
        if self.dist.multi:
            # every rank keeps its stitched pages in HBM; rank 0 receives the slabs over NCCL and writes the file
            local = torch.zeros((hi - lo, h, w), dtype=torch.uint8, device=self.device)
            self.session.predict_stream(source, lo, hi, None, keep=self._keep, progress=progress, out_dev=local)
            full = self.dist.gather_slabs(local, self.dist.shards(self.tif_len))
            if full is not None:
                with tiff.TiffWriter(self.result_name, bigtiff=False) as tif:
                    for frame in full.cpu().numpy():
                        tif.write(frame, contiguous=True)
        else:
            # single process: pages are appended to the result file as the chunks come back (:102,123)
            with tiff.TiffWriter(self.result_name, bigtiff=False) as tif:
                def sink(first, pages):
                    for frame in pages:
                        tif.write(frame, contiguous=True)
                self.session.predict_stream(source, lo, hi, sink, keep=self._keep, progress=progress)
        self.fallback_ops = self.session.engine.fallback_ops
        self.session.close()
        del self.session
        if self._keep is not None:
            self.patches = np.concatenate(self._keep['patches'])
            self.result_patches = np.concatenate(self._keep['result_patches'])
        del self.model_params
        torch.cuda.empty_cache()
