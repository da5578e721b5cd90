#!/usr/bin/env python
"""vvcb_chroma_joint_tu_eval on the GPU: latency of a walk-sized batch (30 chroma CUs x the three TuCResModes, dependent quantisation + rate)
and the throughput of a 1080p 4:2:0 sweep (every aligned 4..32 chroma block, one joint candidate each), with the device time per stage from
torch.profiler's CUDA activity records, the launches of vvcb_chroma_tu_eval on the same walk for comparison, and the card's name and power
limit read in the same run.  Prints one JSON object; --out writes it too.  GPU box only; a measuring aid for profiles/, not a bench line."""
import argparse
import json
import os
import re
import subprocess
import sys
import time
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import vvc_intra_b200 as vb
from vvc_intra_b200 import engine as E
from chroma_eval_probe import sweep_visits
import chroma_tu_probe as TP

# stage of each kernel of the call (vvcb_api.cu, chroma_joint_tu_chunk)
STAGES = (('prediction', r'chroma_tu_pred_kernel'), ('transform', r'tu_eval_kernel'), ('prices', r'rates_from_states_kernel|dq_rate_kernel'),
          ('dq_order', r'dq_first_kernel|dq_hist_kernel|dq_scan_kernel|dq_scatter_kernel'), ('dq', r'dq_kernel<'),
          ('rate', r'rate_kernel<'), ('joint', r'chroma_joint_kernel'))


def stage_ms(fn, calls):
    """device milliseconds per call by stage (and in total), from the profiler's CUDA kernel records"""
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
    out, other = defaultdict(float), defaultdict(float)
    for e in prof.key_averages():
        if e.device_time_total <= 0:
            continue
        name = next((s for s, pat in STAGES if re.search(pat, e.key)), None)
        if name:
            out[name] += e.device_time_total / 1e3 / calls
        else:
            other[e.key[:60]] += e.device_time_total / 1e3 / calls
    out = dict(out)
    out['kernels_total'] = sum(out.values())
    out['other_device_ms'] = dict(other)
    return out


def joint_jobs(visits, modes, qp=32):
    """one joint job per visit and mode (CSign +1), candidate DM, dependent quantisation + rate"""
    n = len(visits) * len(modes)
    jobs = np.zeros(n, E.CHROMA_JOINT_TU_JOB_DTYPE)
    jobs['visit'] = np.repeat(np.arange(len(visits)), len(modes))
    jobs['cand'] = 7
    jobs['mode'] = np.tile(np.array(modes), len(visits))
    jobs['sign'] = 1
    jobs['flags'] = 1 | 2 | 32                                      # VVCB_TU_QUANT | VVCB_TU_DEPQUANT | VVCB_TU_RATE
    jobs['qp_per'], jobs['qp_rem'] = qp // 6, qp % 6
    jobs['lambda'] = 0.57 * 2 ** ((qp - 12) / 3) * 16
    sizes = 2 << (visits['log2w'][jobs['visit']].astype(np.int64) + visits['log2h'][jobs['visit']].astype(np.int64))
    jobs['offset'] = np.concatenate(([0], np.cumsum(sizes)[:-1]))
    return jobs, int(sizes.sum())


def joint_states(rng, n):
    s = np.zeros(n, E.CHROMA_JOINT_CTX_STATES_DTYPE)
    s['chroma'] = TP.states(rng, n)
    jm = s['joint'].view(np.uint16).reshape(n, 3, 3)
    jm[:, :, 0] = rng.integers(1, 0x400, (n, 3)) << 5
    jm[:, :, 1] = rng.integers(1, 0x4000, (n, 3)) << 1
    jm[:, :, 2] = (rng.integers(4, 8, (n, 3)) << 4) | rng.integers(4, 8, (n, 3))
    return s


def timed(eng, run, calls):
    l0 = eng.launch_count
    t0 = time.perf_counter()
    for _ in range(calls):
        run()                                                       # synchronous: returns after the results are on the host
    return (time.perf_counter() - t0) / calls, (eng.launch_count - l0) / calls


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
    st = joint_states(rng, 1)
    with vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=128) as eng:
        eng.frame_begin(luma)
        eng.reco_from_orig()
        eng.chroma_frame_begin(cb, cr)
        eng.chroma_reco_update(cb, cr)
        sweep = sweep_visits(rng, cw, ch)
        # ---- walk: 30 CUs of mixed shapes from the inside of the picture, the three modes each
        inner = np.flatnonzero((sweep['x'] >= 64) & (sweep['y'] >= 64) & (sweep['x'] < cw - 64) & (sweep['y'] < ch - 64))
        walk = sweep[rng.choice(inner, 30, replace=False)]
        wj, wns = joint_jobs(walk, [1, 2, 3])
        run = lambda: eng.chroma_joint_tu_eval(walk, wj, wns, states=st)
        for _ in range(20):
            run()
        dt, launches = timed(eng, run, a.calls)
        # the separate call on the same 90 candidates' CUs and quantiser, for the launch count
        sj, sns = TP.jobs_for(walk, 3, rng)
        sep = lambda: eng.chroma_tu_eval(walk, sj, sns, states=st['chroma'])
        sep()
        sdt, slaunches = timed(eng, sep, 20)
        res['walk'] = dict(cus=len(walk), candidates=len(wj), calls=a.calls, ms_per_call=1e3 * dt, launches_per_call=launches,
                           device_ms_per_call=stage_ms(run, 100), chroma_tu_eval_launches_per_call=slaunches,
                           chroma_tu_eval_ms_per_call=1e3 * sdt)
        # ---- sweep: one joint candidate per block (DM, mode 2), dependent quantisation + rate
        sj, sns = joint_jobs(sweep, [2])
        run = lambda: eng.chroma_joint_tu_eval(sweep, sj, sns, states=st)
        run()
        reps = 5
        dt, launches = timed(eng, run, reps)
        sm = stage_ms(run, reps)
        res['sweep'] = dict(candidates=len(sj), chroma_picture='%dx%d' % (cw, ch), shapes=16, s_per_call=dt, candidates_per_s=len(sj) / dt,
                            launches_per_call=launches, device_ms_per_call=sm,
                            kernel_candidates_per_s=len(sj) / (sm['kernels_total'] * 1e-3),
                            note='a candidate = one chroma CU x one candidate mode x one TuCResMode: both predictions, the combined residual, '
                                 'its transform, dependent quantisation and inverse, the inverse mapping, both reconstructions and SSEs, the '
                                 'cbf and joint-flag bins and residual bits; s_per_call includes the host validation, job building and the '
                                 'copies, device_ms_per_call the kernels by stage (65 536 candidates per chunk)')
    print(json.dumps(res, indent=1))
    if a.out:
        with open(a.out, 'w') as f:
            json.dump(res, f, indent=1)


if __name__ == '__main__':
    main()
