#!/usr/bin/env python
"""Device time of every rmd_eval_kernel<TILE, KIND, MODE> instantiation in bench.py's resident 1080p sweep.

Runs the resident 10-bit 1920x1080 rough-mode-decision sweep (every evaluation slot of every CU of the frame, the workload of bench.py's
`value`) --passes times after --warmup passes, under torch.profiler with CUDA activities, and prints the mean duration per sweep of each
evaluation-kernel instantiation, the sums per prediction kind (angular, planar / DC, MIP) and the list kernel's.  The library's kernels
are found by name in the profiler's kernel records; a run in which the profiler records none of them fails.

    python tools/eval_kernel_times.py [--passes 10] [--warmup 3] [--json OUT]
"""
import argparse
import json
import os
import re
import sys
import tempfile
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

KINDS = ('angular', 'planar_dc', 'mip')                  # KIND_ANG, KIND_PDC, KIND_MIP of vvcb_rmd.cuh
EVAL_RE = re.compile(r'rmd_eval_kernel<(\d), (\d), (\d)>')


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('--passes', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--json', help='also write the result as JSON to this file')
    a = ap.parse_args()
    if a.passes < 1 or a.warmup < 0:
        ap.error('--passes must be at least 1 and --warmup not negative')

    import torch
    from torch.profiler import ProfilerActivity, profile
    import vvc_intra_b200 as vb
    from bench import BITS, CTU, H, W, synth_luma

    if not torch.cuda.is_available():
        sys.exit('eval_kernel_times: no CUDA device')
    torch.zeros(1, device='cuda')                        # the profiler's CUDA activity needs the runtime initialised
    vis = vb.build_sweep_visits(W, H, qp=32, ctu=CTU)
    n = len(vis)
    pitch = (W + 63) & ~63
    plane = np.zeros((H, pitch), np.int16)
    plane[:, :W] = synth_luma(0)
    with vb.IntraCostEngine(device=0, bit_depth=BITS, ctu_size=CTU) as eng:
        d_plane = eng.dev_alloc(plane.nbytes)
        eng.dev_upload(d_plane, plane)
        d_vis = eng.dev_alloc(vis.nbytes)
        eng.dev_upload(d_vis, vis)
        d_res = eng.dev_alloc(n * vb.RESULT_DTYPE.itemsize)
        eng.frame_bind_device(d_plane, d_plane, pitch, W, H)
        for _ in range(a.warmup):
            eng.rmd_eval_device(d_vis, n, d_res, None)
        eng.sync()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(a.passes):
                eng.rmd_eval_device(d_vis, n, d_res, None)
            eng.sync()

    # the kernel records of the trace (the library launches from its own C code, outside any torch operator)
    with tempfile.TemporaryDirectory() as tmp:
        trace = os.path.join(tmp, 'trace.json')
        prof.export_chrome_trace(trace)
        with open(trace) as f:
            events = json.load(f)['traceEvents']
    per_inst = defaultdict(float)                        # (tile, kind, mode) -> total us
    lists_us = 0.0
    for ev in events:
        if ev.get('cat') != 'kernel':
            continue
        name, us = ev.get('name', ''), float(ev.get('dur', 0.0))
        m = EVAL_RE.search(name)
        if m:
            per_inst[tuple(int(g) for g in m.groups())] += us
        elif 'rmd_lists_kernel' in name:
            lists_us += us
    if not per_inst:
        sys.exit('eval_kernel_times: the profiler recorded no rmd_eval_kernel launch')

    rows = [{'tile': t, 'kind': KINDS[k], 'mode': md, 'us_per_sweep': us / a.passes} for (t, k, md), us in sorted(per_inst.items())]
    by_kind = {kind: sum(r['us_per_sweep'] for r in rows if r['kind'] == kind) for kind in KINDS}
    out = {'gpu': torch.cuda.get_device_name(0), 'visits': n, 'passes': a.passes, 'launches_per_sweep': len(rows),
           'kernels': rows, 'us_per_sweep_by_kind': by_kind, 'eval_us_per_sweep': sum(by_kind.values()),
           'lists_us_per_sweep': lists_us / a.passes}
    print('%-26s %12s' % ('rmd_eval_kernel<T,K,M>', 'us / sweep'))
    for r in rows:
        print('%-26s %12.1f' % ('<%d,%d,%d> %s' % (r['tile'], KINDS.index(r['kind']), r['mode'], r['kind']), r['us_per_sweep']))
    for kind in KINDS:
        print('%-26s %12.1f' % ('sum ' + kind, by_kind[kind]))
    print('%-26s %12.1f' % ('sum eval', out['eval_us_per_sweep']))
    print('%-26s %12.1f' % ('rmd_lists_kernel', out['lists_us_per_sweep']))
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(out, f, indent=1)


if __name__ == '__main__':
    main()
