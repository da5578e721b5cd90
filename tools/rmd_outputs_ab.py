#!/usr/bin/env python
"""Compare the rough-mode-decision outputs of two library builds byte for byte.

Each build runs in a process of its own (VVCB_LIBRARY_PATH selects the library) on the same seeded inputs:
  - the full sweep (every CU position and shape) of two synthetic 1920x1080 10-bit frames, at QP 32 and QP 27;
  - the full sweep of a synthetic 416x240 8-bit picture.
Every workload goes through vvcb_rmd_eval with detail tables, so the result records (candidate lists and costs) and the per-slot SAD /
SATD tables are both compared.  The workers hash the arrays in chunks of 4 096 visits; the report names the first chunk that differs.

    python tools/rmd_outputs_ab.py LIB_A LIB_B [--json OUT]
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

CHUNK = 4096
WORKLOADS = (('1080p_10b_f0_qp32', 1920, 1080, 10, 0, 32), ('1080p_10b_f1_qp27', 1920, 1080, 10, 1, 27),
             ('416x240_8b_f0_qp32', 416, 240, 8, 0, 32))


def chunk_hashes(a):
    b = a.view(np.uint8).reshape(len(a), -1)
    return [hashlib.sha256(b[i:i + CHUNK].tobytes()).hexdigest() for i in range(0, len(a), CHUNK)]


def worker(out_path):
    import vvc_intra_b200 as vb
    from make_golden import synth_yuv
    out = {'library': vb.engine.library_path()}
    for name, w, h, bd, frame, qp in WORKLOADS:
        y = synth_yuv(w, h, bd, frame)[0].astype(np.int16)
        vis = vb.build_sweep_visits(w, h, qp=qp, ctu=128)
        with vb.IntraCostEngine(0, bd, 128) as eng:
            eng.frame_begin(y)
            eng.reco_update(y)
            # zero-filled outputs: padding bytes compare equal too
            res, det = eng.rmd_eval(vis, out=np.zeros(len(vis), vb.RESULT_DTYPE), detail_out=np.zeros(len(vis), vb.DETAIL_DTYPE))
        out[name] = {'visits': len(vis), 'result': chunk_hashes(res), 'detail': chunk_hashes(det)}
    with open(out_path, 'w') as f:
        json.dump(out, f)


def main():
    ap = argparse.ArgumentParser(description=__doc__.split('\n')[0])
    ap.add_argument('lib_a')
    ap.add_argument('lib_b')
    ap.add_argument('--json', help='also write the report as JSON to this file')
    ap.add_argument('--worker', help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        worker(a.worker)
        return
    runs = []
    with tempfile.TemporaryDirectory() as tmp:
        for i, lib in enumerate((a.lib_a, a.lib_b)):
            if not os.path.isfile(lib):
                sys.exit('rmd_outputs_ab: no library at %s' % lib)
            path = os.path.join(tmp, 'run%d.json' % i)
            env = dict(os.environ, VVCB_LIBRARY_PATH=os.path.abspath(lib))
            subprocess.check_call([sys.executable, os.path.abspath(__file__), a.lib_a, a.lib_b, '--worker', path], env=env)
            with open(path) as f:
                runs.append(json.load(f))
    report, same = {'lib_a': a.lib_a, 'lib_b': a.lib_b, 'workloads': {}}, True
    for name, *_ in WORKLOADS:
        ra, rb = runs[0][name], runs[1][name]
        entry = {'visits': ra['visits']}
        for field in ('result', 'detail'):
            diff = [i for i, (x, y) in enumerate(zip(ra[field], rb[field])) if x != y]
            ok = ra['visits'] == rb['visits'] and len(ra[field]) == len(rb[field]) and not diff
            entry[field] = 'identical' if ok else 'differ from visit %d' % ((diff[0] if diff else 0) * CHUNK)
            same = same and ok
        report['workloads'][name] = entry
        print('%-20s %7d visits  results: %-28s details: %s' % (name, entry['visits'], entry['result'], entry['detail']))
    report['identical'] = same
    print('IDENTICAL' if same else 'DIFFERENT')
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(report, f, indent=1)
    sys.exit(0 if same else 1)


if __name__ == '__main__':
    main()
