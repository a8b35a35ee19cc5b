#!/usr/bin/env python
"""Cost of test-time augmentation on the cfg 1, cfg 2 and cfg 4 workloads of bench.py (which stays untouched).

For every config the same Session runs the modes tta=None, 'flips' and (2D) 'dihedral' in alternation, `--reps` times
each: device-resident and end-to-end rates, and the device time of the TTA gather and merge launches, taken from CUDA
events around every call of engine.gather_tiles_tta / engine.tta_accumulate in the TTA modes, as a share of the step
(tta=None gathers through the same entry point with transform 0, which is no TTA work). The card's name, power limit
and SM clock are read in the same call. One JSON line per config and mode.

    python tools/bench_tta.py [--configs 1,2,4] [--frames 32] [--reps 2] [--out DIR]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from bio_image_unet_b200 import engine as E  # noqa: E402
from bio_image_unet_b200 import pipeline2d as P  # noqa: E402
from bio_image_unet_b200.dist import DistContext  # noqa: E402

_EVENTS = []
_TTA_ON = [False]          # set while the session runs a TTA mode


def _timed(fn):
    def wrap(*a, **k):
        if not _TTA_ON[0]:
            return fn(*a, **k)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = fn(*a, **k)
        e1.record()
        _EVENTS.append((e0, e1))
        return r
    return wrap


E.gather_tiles_tta = _timed(E.gather_tiles_tta)
E.gather_tiles_f32_tta = _timed(E.gather_tiles_f32_tta)
E.tta_accumulate = _timed(E.tta_accumulate)


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else 'unknown'


def set_tta(ses, mode, dims, channels):
    """Switch an existing Session's tta mode (re-plans on the next call)."""
    tile = ses.resize_dim
    ses.tta = P.tta_codes(mode, dims, tile)
    _TTA_ON[0] = ses.tta is not None
    ses._planner.extra_per_tile = lambda t: P.tta_extra_bytes(mode, channels, t)
    ses._planner.tile = None
    ses._planner.tile_batch = None


def timed(fn, reps):
    torch.cuda.synchronize()
    _EVENTS.clear()
    t0 = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    tta_ms = sum(a.elapsed_time(b) for a, b in _EVENTS) / reps
    return dt, tta_ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--configs', default='1,2,4')
    ap.add_argument('--frames', type=int, default=32, help='cfg-2 frames per step')
    ap.add_argument('--reps', type=int, default=2, help='alternations of the three modes')
    ap.add_argument('--steps', type=int, default=3, help='timed steps per measurement')
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    dev = torch.device('cuda:0')
    ctx = DistContext(False)
    lines = []
    for cfg in [int(c) for c in a.configs.split(',')]:
        args = argparse.Namespace(precision=None, frames=a.frames, chunk_frames=8, add_patch=0, vol=None)
        wl = bench.WORKLOADS[cfg](args, dev, ctx).setup()
        dims = 3 if cfg == 4 else 2
        modes = [None, 'flips'] + (['dihedral'] if dims == 2 else [])
        for m in modes:                                     # warm up every mode's plans and modules
            set_tta(wl.ses, m, dims, 1)
            wl.step_device()
            wl.step_e2e()
        res = {m: [] for m in modes}
        for _ in range(a.reps):
            for m in modes:
                set_tta(wl.ses, m, dims, 1)
                wl.step_device()
                dt_dev, tta_ms = timed(wl.step_device, a.steps)
                dt_e2e, _ = timed(wl.step_e2e, a.steps)
                res[m].append({'device_rate': wl.units_per_step / dt_dev, 'e2e_rate': wl.units_per_step / dt_e2e,
                               'step_ms': dt_dev * 1e3, 'tta_launch_ms': tta_ms,
                               'tta_launch_share': tta_ms / (dt_dev * 1e3), 'card': card()})
        for m in modes:
            line = {'config': cfg, 'workload': wl.name, 'precision': wl.precision, 'tta': m, 'unit': wl.unit,
                    'runs': res[m]}
            print(json.dumps(line), flush=True)
            lines.append(line)
        wl.ses.close()
        del wl
        torch.cuda.empty_cache()
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, 'bench_tta.json'), 'w') as f:
            json.dump(lines, f, indent=1)


if __name__ == '__main__':
    main()
