#!/usr/bin/env python
"""vvcb_isp_eval on the GPU: latency, launches and per-stage kernel time of a walk-sized batch (28 candidates of four CUs, dependent
quantisation and residual rate), and the throughput of a sweep-sized batch (one candidate per in-scope CU position of a 1080p picture,
every in-scope CU shape and split), with the card's name and power limit read in the same run.  Prints one JSON object; --out writes it
too.  GPU box only; a measuring aid for profiles/, not a bench line."""
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

HOR, VER = 1, 2


def blocks(cu_w, cu_h, hor):
    split, other = (cu_h, cu_w) if hor else (cu_w, cu_h)
    size = max(split >> 2, 16 // other if other < 16 else 1)
    return cu_w if hor else size, size if hor else cu_h


def in_scope():
    return [(1 << lw, 1 << lh, isp) for lw in range(2, 7) for lh in range(2, 7) for isp in (HOR, VER)
            if lw + lh > 4 and min(blocks(1 << lw, 1 << lh, isp == HOR)) >= 4]


def states(rng, n):
    s = np.zeros(n, E.CTX_STATES_DTYPE)
    f = s.view(np.uint8).reshape(n, -1).view(np.uint16).reshape(n, -1, 3)
    f[:, :, 0] = rng.integers(1, 0x400, f.shape[:2]) << 5
    f[:, :, 1] = rng.integers(1, 0x4000, f.shape[:2]) << 1
    f[:, :, 2] = (5 << 4) | 8
    return s


def job(rate_idx, visit, isp, mode, qp, off):
    j = np.zeros(1, E.ISP_JOB_DTYPE)[0]
    j['visit'], j['isp_mode'], j['mode'], j['flags'], j['use_mts'], j['max_tb_size'] = visit, isp, mode, 1 | 2 | 32, 1, 64
    j['qp_per'], j['qp_rem'], j['rate_idx'], j['offset'] = qp // 6, qp % 6, rate_idx, off
    for t in range(2):
        j['cbf'][t]['state'] = (0x3000, 0x3000)
        j['cbf'][t]['rate'] = (5 << 4) | 8
    j['lambda'] = 0.57 * 2.0 ** ((qp - 12) / 3.0)
    return j


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=300)
    ap.add_argument('--out')
    a = ap.parse_args()
    rng = np.random.default_rng(1)
    bd, W, H = 10, 1920, 1080
    orig = rng.integers(0, 1024, (H, W)).astype(np.int16)
    res = dict(gpu=subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True, text=True).stdout.strip())
    with vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=128) as eng:
        eng.frame_begin(orig)
        eng.reco_from_orig()
        # ---- walk: four CUs x up to 8 candidates (the in-scope splits x four modes)
        cus = [(16, 16), (32, 16), (8, 32), (32, 32)]
        visits = np.zeros(len(cus), E.VISIT_DTYPE)
        jobs, off = [], 0
        for c, (w, h) in enumerate(cus):
            v = visits[c]
            v['x'], v['y'], v['log2w'], v['log2h'] = 256 + 128 * c, 256, w.bit_length() - 1, h.bit_length() - 1
            v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'], v['flags'] = 1, w // 4, w // 4, h // 4, 0, 3
            for isp in (HOR, VER):
                if min(blocks(w, h, isp == HOR)) < 4:
                    continue
                for mode in (0, 1, 18, 50):
                    jobs.append(job(len(jobs), c, isp, mode, 32, off))
                    off += w * h
        jobs = np.array(jobs, E.ISP_JOB_DTYPE)
        st = states(rng, len(jobs))
        for _ in range(20):
            eng.isp_eval(visits, jobs, off, states=st)
        l0 = eng.launch_count
        t0 = time.perf_counter()
        for _ in range(a.calls):
            eng.isp_eval(visits, jobs, off, states=st)          # synchronous: returns after the device results are on the host
        dt = time.perf_counter() - t0
        launches = (eng.launch_count - l0) / a.calls
        eng.kernel_timing(True)
        eng.tu_kernel_times()
        for _ in range(a.calls):
            eng.isp_eval(visits, jobs, off, states=st)
        ms = eng.tu_kernel_times()
        eng.kernel_timing(False)
        res['walk'] = dict(candidates=len(jobs), cus=len(cus), calls=a.calls, us_per_call=1e6 * dt / a.calls, launches_per_call=launches,
                           kernel_ms_per_call=dict(pred_and_transform=ms[0] / a.calls, quantiser=ms[1] / a.calls,
                                                   reconstruction=ms[2] / a.calls, rate=ms[3] / a.calls))
        # ---- sweep: one candidate per in-scope CU position of the picture (all shapes and splits), mode cycling
        vis, jb, off = [], [], 0
        proto = job(0, 0, HOR, 0, 32, 0)
        for w, h, isp in in_scope():
            ys, xs = np.meshgrid(np.arange(4, H - h + 1, h), np.arange(4, W - w + 1, w), indexing='ij')
            v = np.zeros(ys.size, E.VISIT_DTYPE)
            v['x'], v['y'], v['log2w'], v['log2h'] = xs.ravel(), ys.ravel(), w.bit_length() - 1, h.bit_length() - 1
            v['avail_al'], v['n_above'], v['n_left'], v['flags'] = 1, w // 4, h // 4, 3
            j = np.repeat(np.array([proto], E.ISP_JOB_DTYPE), ys.size)
            first = sum(len(a) for a in vis)
            j['visit'] = first + np.arange(ys.size)
            j['isp_mode'], j['mode'], j['rate_idx'] = isp, (first + np.arange(ys.size)) % 67, (first + np.arange(ys.size)) % 64
            j['offset'] = off + w * h * np.arange(ys.size)
            off += w * h * ys.size
            vis.append(v)
            jb.append(j)
        vis, jb = np.concatenate(vis), np.concatenate(jb)
        st = states(rng, 64)
        eng.isp_eval(vis, jb, off, states=st)
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            eng.isp_eval(vis, jb, off, states=st)
        dt = (time.perf_counter() - t0) / reps
        res['sweep'] = dict(candidates=len(jb), picture='%dx%d' % (W, H), shapes=len(in_scope()), s_per_call=dt,
                            candidates_per_s=len(jb) / dt, note='host-to-device copies, validation and job building included')
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
