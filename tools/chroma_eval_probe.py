#!/usr/bin/env python
"""vvcb_chroma_eval on the GPU: latency of a walk-sized batch (30 chroma CUs, all 8 candidates, LM modes on) and the throughput of a
1080p 4:2:0 sweep (every aligned 4..32 chroma block), with the device time of chroma_eval_kernel from torch.profiler's CUDA activity
records and the card's name and power limit read in the same run.  Prints one JSON object; --out writes it too.  GPU box only; a
measuring aid for profiles/, not a bench line."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vvc_intra_b200 as vb
from vvc_intra_b200 import engine as E

SHAPES = [(1 << a, 1 << b) for a in range(2, 6) for b in range(2, 6)]


def sweep_visits(rng, cw, ch):
    """every aligned 4..32 block of the chroma picture, full availability where the picture has the neighbours"""
    out = []
    for w, h in SHAPES:
        ys, xs = np.meshgrid(np.arange(0, ch - h + 1, h), np.arange(0, cw - w + 1, w), indexing='ij')
        v = np.zeros(ys.size, E.CHROMA_VISIT_DTYPE)
        x, y = xs.ravel(), ys.ravel()
        v['x'], v['y'], v['log2w'], v['log2h'] = x, y, w.bit_length() - 1, h.bit_length() - 1
        v['avail_al'] = (x > 0) & (y > 0)
        v['n_above'], v['n_left'] = np.where(y > 0, w // 2, 0), np.where(x > 0, h // 2, 0)
        v['n_above_right'] = np.where(y > 0, np.clip((cw - x - w) // 2, 0, w // 2), 0)
        v['n_below_left'] = np.where(x > 0, np.clip((ch - y - h) // 2, 0, h // 2), 0)
        out.append(v)
    v = np.concatenate(out)
    v['dm_mode'] = rng.integers(0, 67, len(v))
    v['cclm'] = 1
    return v


def kernel_ms(fn, calls):
    """device milliseconds per call of chroma_eval_kernel, from the profiler's CUDA kernel records"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
    us = sum(e.device_time_total for e in prof.key_averages() if 'chroma_eval_kernel' in e.key)
    return us / 1e3 / calls


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=300)
    ap.add_argument('--out')
    a = ap.parse_args()
    rng = np.random.default_rng(1)
    bd, W, H = 10, 1920, 1080
    cw, ch = W // 2, H // 2
    luma = rng.integers(0, 1024, (H, W)).astype(np.int16)
    cb, cr = (rng.integers(0, 1024, (ch, cw)).astype(np.int16) for _ in range(2))
    res = dict(gpu=subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout.strip())
    with vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=128) as eng:
        eng.frame_begin(luma)
        eng.reco_from_orig()
        eng.chroma_frame_begin(cb, cr)
        eng.chroma_reco_update(cb, cr)
        sweep = sweep_visits(rng, cw, ch)
        # ---- walk: 30 CUs of mixed shapes from the inside of the picture
        inner = np.flatnonzero((sweep['x'] >= 64) & (sweep['y'] >= 64) & (sweep['x'] < cw - 64) & (sweep['y'] < ch - 64))
        walk = sweep[rng.choice(inner, 30, replace=False)]
        for _ in range(20):
            eng.chroma_eval(walk)
        l0 = eng.launch_count
        t0 = time.perf_counter()
        for _ in range(a.calls):
            eng.chroma_eval(walk)                    # synchronous: returns after the results are on the host
        dt = time.perf_counter() - t0
        res['walk'] = dict(visits=len(walk), calls=a.calls, ms_per_call=1e3 * dt / a.calls, launches_per_call=(eng.launch_count - l0) / a.calls,
                           kernel_ms_per_call=kernel_ms(lambda: eng.chroma_eval(walk), 100))
        # ---- sweep
        eng.chroma_eval(sweep)
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            eng.chroma_eval(sweep)
        dt = (time.perf_counter() - t0) / reps
        kms = kernel_ms(lambda: eng.chroma_eval(sweep), reps)
        n_eval = int(len(sweep) * 16)
        res['sweep'] = dict(visits=len(sweep), chroma_picture='%dx%d' % (cw, ch), shapes=len(SHAPES), s_per_call=dt,
                            visits_per_s=len(sweep) / dt, candidate_evaluations_per_s=n_eval / dt,
                            kernel_ms_per_call=kms, kernel_visits_per_s=len(sweep) / (kms * 1e-3),
                            kernel_candidate_evaluations_per_s=n_eval / (kms * 1e-3),
                            note='a candidate evaluation = one candidate of one component (8 x Cb / Cr per visit): prediction, SAD, SATD; '
                                 's_per_call includes the host validation and the copies, kernel_* the kernel alone')
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
