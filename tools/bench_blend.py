#!/usr/bin/env python
"""Cost of the Gaussian overlap blend (blend='gaussian') against the reference's stitches, on the cfg 2 and cfg 4
geometries of bench.py (which stays untouched). The card's name, power limit and SM clock are read in the same call.

1. Kernels, CUDA events over `--launches` launches after warm-up, each stitch timed twice:
   - 'l2_warm': back to back, so whatever of the working set fits the 126 MB L2 stays there;
   - 'l2_cold': one launch at a time, a 512 MiB buffer overwritten before each (a cold L2).
   cfg 2 chunk: 8 frames of 2048^2, 512^2 tiles, add_tile=1 (200 tiles): stitch_mean_u8 vs stitch_weighted_u8.
   cfg 4 volume: 256 x 1024 x 1024, 64 x 128 x 128 patches, add_patch 0 (256 patches): stitch_mod3_u8 vs
   stitch_weighted_u8. Rates are algorithmic bytes (every tile byte read once, every output byte written once) over
   the time, and that rate's share of the HBM3e data-sheet bandwidth of 7.7 TB/s.
2. unet.Session.predict_movie on the device-resident cfg 2 movie, blend None and 'gaussian' alternated `--reps` times.

One JSON line per measurement.

    python tools/bench_blend.py [--launches 200] [--frames 64] [--reps 3] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from bio_image_unet_b200 import engine as E  # noqa: E402
from bio_image_unet_b200 import pipeline2d as P  # noqa: E402
from bio_image_unet_b200 import tiling  # noqa: E402
from bio_image_unet_b200.dist import DistContext  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def time_kernel(fn, launches, flush):
    for _ in range(10):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(launches):
        fn()
    e1.record()
    torch.cuda.synchronize()
    warm = e0.elapsed_time(e1) / launches
    evs = []
    for _ in range(launches):
        flush.add_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    cold = sum(a.elapsed_time(b) for a, b in evs) / launches
    return warm, cold


def kernel_lines(launches):
    dev = torch.device('cuda:0')
    flush = torch.zeros(512 << 20, dtype=torch.uint8, device=dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    out = []
    # cfg 2 chunk
    f, (h, w), rd = 8, (2048, 2048), (512, 512)
    n_x, n_y, xs, ys = tiling.grid_2d(h, w, rd, 1)
    tiles = torch.randint(0, 256, (f * n_x * n_y, 1, *rd), dtype=torch.uint8, device=dev, generator=gen)
    mean = E.stitch_mean_u8(tiles, f, 1, (h, w), xs, ys, rd)
    tables = P.blend_tables(rd)
    unit = E.stitch_weighted_u8(tiles, f, 1, (1, h, w), [0], xs, ys, (1, *rd), [1], [1] * rd[0], [1] * rd[1])
    assert torch.equal(unit.view(mean.shape), mean)
    nbytes = tiles.numel() + mean.numel()
    cases = [('cfg2_chunk', 'stitch_mean_u8', lambda: E.stitch_mean_u8(tiles, f, 1, (h, w), xs, ys, rd)),
             ('cfg2_chunk', 'stitch_weighted_u8',
              lambda: E.stitch_weighted_u8(tiles, f, 1, (1, h, w), [0], xs, ys, (1, *rd), *tables))]
    geo = {'cfg2_chunk': dict(frames=f, frame=[h, w], tile=list(rd), add_tile=1, tiles=int(tiles.shape[0]),
                              bytes=int(nbytes))}
    # cfg 4 volume
    vol, patch = (256, 1024, 1024), (64, 128, 128)
    n_z, n_x3, n_y3, zs, xs3, ys3 = tiling.grid_3d(vol, patch, 0)
    tiles3 = torch.randint(0, 256, (n_z * n_x3 * n_y3, *patch), dtype=torch.uint8, device=dev, generator=gen)
    tables3 = P.blend_tables(patch)
    nbytes3 = tiles3.numel() + int(np.prod(vol))
    cases += [('cfg4_volume', 'stitch_mod3_u8', lambda: E.stitch_mod3_u8(tiles3, vol, zs, xs3, ys3, patch)),
              ('cfg4_volume', 'stitch_weighted_u8',
               lambda: E.stitch_weighted_u8(tiles3, 1, 1, vol, zs, xs3, ys3, patch, *tables3))]
    geo['cfg4_volume'] = dict(volume=list(vol), patch=list(patch), add_patch=0, tiles=int(tiles3.shape[0]),
                              bytes=int(nbytes3))
    for name, kernel, fn in cases:
        warm, cold = time_kernel(fn, launches, flush)
        nb = geo[name]['bytes']
        line = {'bench': 'stitch_kernel', 'geometry': name, 'kernel': kernel, 'launches': launches, **geo[name],
                'ms_l2_warm': warm, 'ms_l2_cold': cold,
                'gbps_l2_warm': nb / warm / 1e6, 'gbps_l2_cold': nb / cold / 1e6,
                'hbm_share_l2_cold': nb / (cold * 1e-3) / HBM_BYTES_PER_S, 'card': card()}
        print(json.dumps(line), flush=True)
        out.append(line)
    return out


def movie_lines(frames, reps, steps):
    dev = torch.device('cuda:0')
    args = argparse.Namespace(precision=None, frames=frames, chunk_frames=8, add_patch=0, vol=None)
    wl = bench.WORKLOADS[2](args, dev, DistContext(False)).setup()
    ses = wl.ses
    out_dev = torch.empty((frames, 1, *wl.FRAME), dtype=torch.uint8, device=dev)
    results = {}

    def step():
        ses.predict_movie(wl.dev, chunk_frames=wl.chunk, out_dev=out_dev)

    for blend in (None, 'gaussian'):                    # warm up both stitches and the plan
        ses.blend = blend
        step()
        results[blend] = {'runs': [], 'out': None}
    for _ in range(reps):
        for blend in (None, 'gaussian'):
            ses.blend = blend
            step()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / steps
            results[blend]['runs'].append({'step_ms': dt * 1e3, 'mpix_per_s': wl.units_per_step / dt, 'card': card()})
    lines = []
    for blend in (None, 'gaussian'):
        line = {'bench': 'predict_movie', 'workload': wl.name, 'precision': wl.precision, 'frames': frames,
                'chunk_frames': wl.chunk, 'blend': blend, 'steps': steps, 'runs': results[blend]['runs']}
        print(json.dumps(line), flush=True)
        lines.append(line)
    ses.close()
    return lines


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--launches', type=int, default=200)
    ap.add_argument('--frames', type=int, default=64, help='cfg-2 movie frames')
    ap.add_argument('--reps', type=int, default=3, help='alternations of blend None / gaussian')
    ap.add_argument('--steps', type=int, default=3, help='timed predict_movie calls per measurement')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_blend.py measures on a CUDA device and found none')
    print(json.dumps({'card': card()}), flush=True)
    lines = kernel_lines(a.launches)
    torch.cuda.empty_cache()
    lines += movie_lines(a.frames, a.reps, a.steps)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'bench_blend.jsonl'), 'w') as f:
            for line in lines:
                f.write(json.dumps(line) + '\n')


if __name__ == '__main__':
    main()
