#!/usr/bin/env python
"""Generates the committed golden fixtures under tests/golden/ by running the UNMODIFIED reference
encoder (oracle/_ref/EncoderAppTrace, see oracle/Makefile.ref + oracle/ref_trace_hooks.cpp) on
synthetic YUV input (SURVEY.md App. G).  Runs only in the build container (/root/reference present).

    python tools/make_golden.py            # regenerate all fixtures
"""
import gzip
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_CFG = '/root/reference/VVC_project/bin/vs15/msvc-19.16/x86_64/release/encoder_intra.cfg'


def synth_yuv(w, h, bits, frame=0):
    """SURVEY.md 8d / App. G generator (seed 1234 + frame, x shifted by 3*frame, 10-bit = constants x4)."""
    k = 4 if bits == 10 else 1
    rng = np.random.default_rng(1234 + frame)
    y, x = np.mgrid[0:h, 0:w]
    x = x + 3 * frame
    mx = (1 << bits) - 1
    Y = (128 * k + 60 * k * np.sin(x / 37.0) + 40 * k * np.cos(y / 23.0) + ((x // 32 + y // 32) % 2) * 25 * k
         + rng.normal(0, 6 * k, (h, w))).clip(0, mx)
    U = (128 * k + 30 * k * np.sin(x[::2, ::2] / 50.0) + rng.normal(0, 3 * k, (h // 2, w // 2))).clip(0, mx)
    V = (128 * k + 30 * k * np.cos(y[::2, ::2] / 40.0) + rng.normal(0, 3 * k, (h // 2, w // 2))).clip(0, mx)
    dt = np.uint8 if bits == 8 else '<u2'
    return Y.astype(dt), U.astype(dt), V.astype(dt)


def run(name, w, h, bits, qp, env, extra=()):
    tmp = tempfile.mkdtemp(prefix='vvcgold_')
    try:
        Y, U, V = synth_yuv(w, h, bits)
        open(os.path.join(tmp, 'in.yuv'), 'wb').write(Y.tobytes() + U.tobytes() + V.tobytes())
        shutil.copy(REF_CFG, os.path.join(tmp, 'encoder_intra.cfg'))
        open(os.path.join(tmp, 'Time_python.dat'), 'w').close()   # encmain.cpp:195 fclose(NULL) otherwise
        e = dict(os.environ, VVC_TRACE_OUT=os.path.join(tmp, 'trace.bin'), **{k: str(v) for k, v in env.items()})
        cmd = [os.path.join(ROOT, 'oracle/_ref/EncoderAppTrace'), '-c', 'encoder_intra.cfg', '-i', 'in.yuv', '-wdt', str(w),
               '-hgt', str(h), '-q', str(qp), '-f', '1', '-fr', '30', '-b', 'out.bin', '-o', 'rec.yuv',
               '--InputBitDepth=%d' % bits, '--InternalBitDepth=%d' % bits, '--OutputBitDepth=%d' % bits,
               '--SEIDecodedPictureHash=1'] + list(extra)
        out = subprocess.run(cmd, cwd=tmp, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        poc = [l for l in out.stdout.splitlines() if l.startswith('POC')]
        if out.returncode or not poc:
            print(out.stdout[-3000:])
            raise SystemExit('reference encoder failed')
        raw = open(os.path.join(tmp, 'trace.bin'), 'rb').read()
        dst = os.path.join(ROOT, 'tests/golden', name + '.bin.gz')
        with gzip.GzipFile(dst, 'wb', compresslevel=9, mtime=0) as f:
            f.write(raw)
        bs = hashlib.md5(open(os.path.join(tmp, 'out.bin'), 'rb').read()).hexdigest()
        line = '%s: %dx%d %d-bit qp%d %s | %s | bitstream md5 %s | trace %d B -> %d B gz' % (
            name, w, h, bits, qp, ' '.join(extra), poc[0].strip(), bs, len(raw), os.path.getsize(dst))
        print(line)
        return line
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


def main():
    os.makedirs(os.path.join(ROOT, 'tests/golden'), exist_ok=True)
    lines = []
    if len(sys.argv) > 1 and sys.argv[1] == '--extra':
        return extra_fixtures(sys.argv[2:])
    # RMD visits (reference lines, predictions, SAD/SATD, mode bits, candidate lists) + sampled TU records
    lines.append(run('ref_8b_128x64_qp32', 128, 64, 8, 32,
                     dict(VVC_TRACE_VISIT_FIRST=3, VVC_TRACE_VISIT_STRIDE=60, VVC_TRACE_FULL_PRED=1,
                          VVC_TRACE_TU_FIRST=2, VVC_TRACE_TU_STRIDE=400)))
    lines.append(run('ref_10b_192x128_qp27', 192, 128, 10, 27,
                     dict(VVC_TRACE_VISIT_FIRST=2, VVC_TRACE_VISIT_STRIDE=400, VVC_TRACE_FULL_PRED=0,
                          VVC_TRACE_TU_FIRST=1, VVC_TRACE_TU_STRIDE=3000)))
    # scalar-quantiser path (DepQuant / RDOQ off) for the transform+quant kernel
    lines.append(run('ref_10b_64x64_qp32_scalarq', 64, 64, 10, 32,
                     dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000, VVC_TRACE_MAX_VISITS=0,
                          VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=150),
                     extra=['--DepQuant=0', '--RDOQ=0', '--RDOQTS=0', '--SignHideFlag=0']))
    open(os.path.join(ROOT, 'tests/golden/MANIFEST.txt'), 'w').write(
        'Golden fixtures captured from the unmodified reference encoder by tools/make_golden.py\n' + '\n'.join(lines) + '\n')


def extra_fixtures(which):
    """Fixtures added after the first set; each is generated on its own (python tools/make_golden.py --extra NAME...) and
    appended to MANIFEST.txt so that the earlier files keep their bytes."""
    todo = {
        # a16: EncCu::updateCtuDataISlice runs only under rate control (EL/EncGOP.cpp:1565); ragged CTUs (72 wide, 8 high)
        'ref_10b_200x136_ctuhad': lambda n: run(n, 200, 136, 10, 32, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                         VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=0, VVC_TRACE_TU_STRIDE=100000000),
                                                    extra=['--RateControl=1', '--TargetBitrate=400000']),
        # a13: dependent quantisation (DepQuant on as shipped): coefficients, context prices and levels of sampled TUs
        'ref_10b_128x128_qp27_depquant': lambda n: run(n, 128, 128, 10, 27, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                                 VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=900, VVC_TRACE_ONLY='D')),
        'ref_8b_128x64_qp37_depquant': lambda n: run(n, 128, 64, 8, 37, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                             VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=500, VVC_TRACE_ONLY='D')),
        # a13: RDOQ of transform-skip TUs (RDOQTS on as shipped)
        'ref_10b_128x128_qp27_rdoqts': lambda n: run(n, 128, 128, 10, 27, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                               VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=40, VVC_TRACE_ONLY='T')),
        'ref_8b_128x64_qp37_rdoqts': lambda n: run(n, 128, 64, 8, 37, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                           VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=20, VVC_TRACE_ONLY='T')),
        # f1: LFNST (forward after the primary transform, inverse before it) with dependent quantisation
        'ref_10b_128x128_qp27_lfnst': lambda n: run(n, 128, 128, 10, 27, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                              VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=2, VVC_TRACE_TU_STRIDE=700, VVC_TRACE_ONLY='FJ')),
        'ref_8b_128x64_qp32_lfnst': lambda n: run(n, 128, 64, 8, 32, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                          VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=2, VVC_TRACE_TU_STRIDE=400, VVC_TRACE_ONLY='FJ')),
        # f2: residual rate estimation -- CABACWriter::residual_coding on the bit estimator (context states in, fractional bits out)
        'ref_10b_128x128_qp27_resbits': lambda n: run(n, 128, 128, 10, 27, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                                VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=700, VVC_TRACE_ONLY='C')),
        'ref_8b_128x64_qp22_resbits': lambda n: run(n, 128, 64, 8, 22, dict(VVC_TRACE_VISIT_FIRST=0, VVC_TRACE_VISIT_STRIDE=1000000,
                                                                            VVC_TRACE_MAX_VISITS=0, VVC_TRACE_TU_FIRST=3, VVC_TRACE_TU_STRIDE=900, VVC_TRACE_ONLY='C')),
    }
    with open(os.path.join(ROOT, 'tests/golden/MANIFEST.txt'), 'a') as f:
        for n in which or sorted(todo):
            f.write(todo[n](n) + '\n')


# The pictures the reference encoder encodes in the served-encoder tests of tests/test_gpu_parity.py (name: w, h, bits, qp, frame).
SERVED_WORKLOADS = {
    'rmd_8b_128x64_qp32_f0': (128, 64, 8, 32, 0), 'rmd_10b_128x128_qp27_f0': (128, 128, 10, 27, 0),
    'rmd_10b_128x128_qp37_f0': (128, 128, 10, 37, 0), 'rmd_10b_128x128_qp22_f0': (128, 128, 10, 22, 0),
    'rmd_10b_128x64_qp27_f1': (128, 64, 10, 27, 1), 'rmd_10b_128x128_qp32_f2': (128, 128, 10, 32, 2),
    'rmd_10b_128x64_qp37_f3': (128, 64, 10, 37, 3), 'rmd_10b_128x64_qp32_f2': (128, 64, 10, 32, 2),
    'rmd_8b_416x240_qp32_f0': (416, 240, 8, 32, 0),
}


def served_fixture(name, keep=10):
    """tests/golden/served/<name>.bin.gz: the V/R/P/B/L records (reference lines, predictions, SAD/SATD, mode bits, candidate lists)
    of `keep` evenly spaced ones of every 97th rough-mode-decision visit of one picture; the TU records are dropped to keep the file small."""
    import struct
    w, h, bits, qp, frame = SERVED_WORKLOADS[name]
    tmp = tempfile.mkdtemp(prefix='vvcgold_')
    try:
        Y, U, V = synth_yuv(w, h, bits, frame)
        open(os.path.join(tmp, 'in.yuv'), 'wb').write(Y.tobytes() + U.tobytes() + V.tobytes())
        open(os.path.join(tmp, 'Time_python.dat'), 'w').close()
        cfg = os.path.join(ROOT, 'oracle/_ref/encoder_intra.cfg')
        e = dict(os.environ, VVC_TRACE_OUT=os.path.join(tmp, 'trace.bin'), VVC_TRACE_VISIT_FIRST='0', VVC_TRACE_VISIT_STRIDE='97',
                 VVC_TRACE_FULL_PRED='0', VVC_TRACE_TU_FIRST='1000000000', VVC_TRACE_TU_STRIDE='1000000000')
        cmd = [os.path.join(ROOT, 'oracle/_ref/EncoderAppTrace'), '-c', cfg, '-i', 'in.yuv', '-wdt', str(w), '-hgt', str(h), '-q', str(qp),
               '-f', '1', '-fr', '30', '-b', 'out.bin', '--InputBitDepth=%d' % bits, '--InternalBitDepth=%d' % bits, '--OutputBitDepth=%d' % bits]
        out = subprocess.run(cmd, cwd=tmp, env=e, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if out.returncode:
            raise SystemExit('reference encoder failed: ' + out.stdout[-2000:])
        b = open(os.path.join(tmp, 'trace.bin'), 'rb').read()
        visits, o = [], 0
        while o < len(b):
            tag, n = chr(b[o]), struct.unpack_from('<I', b, o + 1)[0]
            if tag == 'V':
                visits.append([])
            if tag in 'VRPBL':
                visits[-1].append(b[o:o + 5 + n])
            o += 5 + n
        pick = np.linspace(0, len(visits) - 1, keep).astype(int)
        dst = os.path.join(ROOT, 'tests/golden/served', name + '.bin.gz')
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        with gzip.GzipFile(dst, 'wb', compresslevel=9, mtime=0) as f:
            f.write(b''.join(r for i in pick for r in visits[i]))
        return '%s: %dx%d %d-bit qp%d frame %d, visits %s of %d' % (name, w, h, bits, qp, frame, pick.tolist(), len(visits))
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
    if len(sys.argv) > 1 and sys.argv[1] == '--served':
        from multiprocessing import Pool
        with Pool(8) as p:
            lines = p.map(served_fixture, sys.argv[2:] or sorted(SERVED_WORKLOADS))
        with open(os.path.join(ROOT, 'tests/golden/MANIFEST.txt'), 'a') as f:
            f.write(''.join('served/' + l + '\n' for l in lines))
        sys.exit(0)
    sys.exit(main())
