"""CPU tests of the host logic above the C ABI: the substituting shim inside the unmodified reference encoder
(oracle/ref_gpu_serve.cpp -> oracle/_ref/EncoderAppServe), its prefetch cache, and the shared-memory broker
(vvc_intra_b200/csrc/vvcb_broker.inc), all running against the ORACLE-BACKED stand-in of the library
(tests/fake_engine, test infrastructure) because this container has no GPU.  The same binaries run against the real
library in tests/test_gpu_parity.py (-m gpu)."""
import ctypes as C
import json
import os
import re
import subprocess
import time

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, 'oracle/_ref')
FAKE = os.path.join(ROOT, 'tests/fake_engine')


@pytest.fixture(scope='module')
def libraries():
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope='module')
def built(libraries):
    need = [os.path.join(REF, f) for f in ('EncoderApp', 'EncoderAppServe', 'encoder_intra.cfg')] + [os.path.join(FAKE, 'libvvc_intra_b200.so'), os.path.join(FAKE, 'vvcb_broker')]
    if not all(os.path.exists(p) for p in need):
        pytest.skip('oracle/_ref binaries are built only in the container that has /root/reference')
    return True


def encoder_args(w, h, bits, qp):
    return ['-c', os.path.join(REF, 'encoder_intra.cfg'), '-i', 'in.yuv', '-wdt', str(w), '-hgt', str(h), '-q', str(qp), '-f', '1', '-fr', '30',
            '--InputBitDepth=%d' % bits, '--InternalBitDepth=%d' % bits, '--OutputBitDepth=%d' % bits]


def write_input(d, w, h, bits, frame=0):
    from make_golden import synth_yuv
    Y, U, V = synth_yuv(w, h, bits, frame)
    (d / 'in.yuv').write_bytes(Y.tobytes() + U.tobytes() + V.tobytes())
    (d / 'Time_python.dat').write_bytes(b'')


def run(cmd, cwd, env=None):
    r = subprocess.run(cmd, cwd=cwd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout[-3000:]
    return r.stdout


def test_broker_header_symbols_are_exported(libraries):
    hdr = open(os.path.join(ROOT, 'include/vvc_intra_b200_broker.h')).read()
    names = sorted(set(re.findall(r'\b(vvcb_broker_[a-z_]+)\s*\(', hdr)))
    assert names == ['vvcb_broker_read_stats', 'vvcb_broker_serve', 'vvcb_broker_stop']
    for lib in (os.path.join(ROOT, 'vvc_intra_b200/libvvc_intra_b200.so'), os.path.join(FAKE, 'libvvc_intra_b200.so')):
        L = C.CDLL(lib)
        for n in names + ['vvcb_cu_eval', 'vvcb_frame_alloc', 'vvcb_orig_update', 'vvcb_reco_update_rects']:
            assert hasattr(L, n), (lib, n)


def test_served_encoder_is_bit_identical_and_computes_nothing_itself(built, tmp_path):
    """The substituting shim: every luma whole-CU prediction, SAD / SATD, transform, quantisation, reconstruction, SSE and residual bit
    count inside estIntraPredLumaQT comes from the engine (here: its oracle-backed stand-in); the bitstream must equal the plain
    encoder's byte for byte, with no candidate fetched on demand and no stale context (the prefetch reaches what the loop asks for)."""
    w, h, bits, qp = 128, 64, 8, 32
    write_input(tmp_path, w, h, bits)
    run([os.path.join(REF, 'EncoderApp')] + encoder_args(w, h, bits, qp) + ['-b', 'plain.bin'], tmp_path)
    env = dict(os.environ, LD_LIBRARY_PATH=FAKE, VVCB_SHIM_REPORT=str(tmp_path / 'rep.json'))
    env.pop('VVCB_BROKER', None)
    run([os.path.join(REF, 'EncoderAppServe')] + encoder_args(w, h, bits, qp) + ['-b', 'serve.bin'], tmp_path, env)
    a, b = (tmp_path / 'plain.bin').read_bytes(), (tmp_path / 'serve.bin').read_bytes()
    assert len(a) > 100 and a == b
    rep = json.loads((tmp_path / 'rep.json').read_text())
    assert rep['enabled'] == 1 and rep['visits'] > 1000 and rep['rmd_round_trips'] == rep['visits']
    assert rep['tu_round_trips'] < 0.05 * rep['visits']                     # ONE round trip per CU: lists and every candidate of all passes (templates)
    assert rep['demand_round_trips'] == 0 and rep['stale_context'] == 0 and rep['tu_residual_bits_reference'] == 0
    assert rep['predictions_skipped'] > 40 * rep['visits'] and rep['distortions_served'] == 2 * rep['predictions_skipped']
    assert rep['tu_quantised'] > 10000 and rep['tu_rdoq_ts'] > 500 and rep['tu_lfnst'] > 2000 and rep['tu_sse'] == rep['tu_quantised']
    assert rep['tu_residual_bits'] > 5000 and rep['tu_preselections'] > 2000


def test_two_round_trips_name_the_same_candidates(built, tmp_path):
    """VVCB_SHIM_TWO_TRIPS: lists first, then the candidates named by the shim from those lists -- the same candidates the engine's template expansion
    names in one round trip (vvcb_expand.inc), the same bitstream."""
    w, h, bits, qp = 64, 64, 8, 27
    write_input(tmp_path, w, h, bits)
    run([os.path.join(REF, 'EncoderApp')] + encoder_args(w, h, bits, qp) + ['-b', 'plain.bin'], tmp_path)
    reps = []
    for k, extra in enumerate(({}, {'VVCB_SHIM_TWO_TRIPS': '1'})):
        env = dict(os.environ, LD_LIBRARY_PATH=FAKE, VVCB_SHIM_REPORT=str(tmp_path / ('rep%d.json' % k)), **extra)
        env.pop('VVCB_BROKER', None)
        run([os.path.join(REF, 'EncoderAppServe')] + encoder_args(w, h, bits, qp) + ['-b', 'serve%d.bin' % k], tmp_path, env)
        assert (tmp_path / 'plain.bin').read_bytes() == (tmp_path / ('serve%d.bin' % k)).read_bytes()
        reps.append(json.loads((tmp_path / ('rep%d.json' % k)).read_text()))
    assert reps[0]['jobs_prefetched'] == reps[1]['jobs_prefetched'] and reps[0]['demand_round_trips'] == reps[1]['demand_round_trips'] == 0
    assert reps[1]['tu_round_trips'] >= reps[1]['visits'] > 10 * (reps[0]['tu_round_trips'] + 1)


def test_prefetch_is_only_a_hint(built, tmp_path):
    """Without any prefetch every candidate is fetched on demand -- slower, same bitstream: speculation never decides a result."""
    w, h, bits, qp = 64, 64, 8, 37
    write_input(tmp_path, w, h, bits)
    run([os.path.join(REF, 'EncoderApp')] + encoder_args(w, h, bits, qp) + ['-b', 'plain.bin'], tmp_path)
    env = dict(os.environ, LD_LIBRARY_PATH=FAKE, VVCB_SHIM_REPORT=str(tmp_path / 'rep.json'), VVCB_SHIM_NO_PREFETCH='1')
    env.pop('VVCB_BROKER', None)
    run([os.path.join(REF, 'EncoderAppServe')] + encoder_args(w, h, bits, qp) + ['-b', 'serve.bin'], tmp_path, env)
    assert (tmp_path / 'plain.bin').read_bytes() == (tmp_path / 'serve.bin').read_bytes()
    rep = json.loads((tmp_path / 'rep.json').read_text())
    assert rep['tu_round_trips'] == 0 and rep['demand_round_trips'] > rep['visits'] and rep['jobs_prefetched'] == 0


def test_broker_batches_several_encoders(built, tmp_path):
    """Three encoder processes (different pictures, different QPs) share one engine context through the broker; every bitstream is
    byte-identical to its plain encoder's and the server merged requests of different clients into one engine batch."""
    cases = [(64, 64, 8, 32, 0), (64, 64, 8, 27, 1), (128, 64, 8, 37, 2)]
    path = str(tmp_path / 'broker.shm')
    server = subprocess.Popen([os.path.join(FAKE, 'vvcb_broker'), path, '--bit-depth', '8', '--clients', '4', '--frame', '128x64', '--workers', '2'],
                              env=dict(os.environ, LD_LIBRARY_PATH=FAKE), stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    try:
        procs = []
        for i, (w, h, bits, qp, frame) in enumerate(cases):
            d = tmp_path / ('c%d' % i)
            d.mkdir()
            write_input(d, w, h, bits, frame)
            run([os.path.join(REF, 'EncoderApp')] + encoder_args(w, h, bits, qp) + ['-b', 'plain.bin'], d)
            env = dict(os.environ, LD_LIBRARY_PATH=FAKE, VVCB_BROKER=path, VVCB_SHIM_REPORT=str(d / 'rep.json'))
            procs.append((d, subprocess.Popen([os.path.join(REF, 'EncoderAppServe')] + encoder_args(w, h, bits, qp) + ['-b', 'serve.bin'], cwd=d, env=env,
                                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for d, p in procs:
            out, _ = p.communicate(timeout=600)
            assert p.returncode == 0, out[-3000:]
            assert (d / 'plain.bin').read_bytes() == (d / 'serve.bin').read_bytes()
            assert json.loads((d / 'rep.json').read_text())['demand_round_trips'] == 0
        stats = json.loads(subprocess.check_output([os.path.join(FAKE, 'vvcb_broker'), path, '--stats'], env=dict(os.environ, LD_LIBRARY_PATH=FAKE)))
        assert stats['clients_seen'] == 3 and stats['max_batch'] >= 2 and stats['visits'] > 1000 and stats['tu_jobs'] > 10000
        assert stats['cycles'] < stats['requests']                           # requests of different clients shared engine batches
    finally:
        subprocess.run([os.path.join(FAKE, 'vvcb_broker'), path, '--stop'], env=dict(os.environ, LD_LIBRARY_PATH=FAKE))
        try:
            server.wait(timeout=30)
        except subprocess.TimeoutExpired:
            server.kill()
    assert server.returncode == 0


def test_broker_rejects_what_does_not_fit(built, tmp_path):
    """A client whose picture exceeds the server's cell, or whose bit depth differs, fails loudly at frame begin / connect."""
    path = str(tmp_path / 'broker.shm')
    env = dict(os.environ, LD_LIBRARY_PATH=FAKE)
    server = subprocess.Popen([os.path.join(FAKE, 'vvcb_broker'), path, '--bit-depth', '8', '--clients', '2', '--frame', '64x64'], env=env)
    try:
        for _ in range(200):
            if os.path.exists(path):
                break
            time.sleep(0.05)
        w, h, bits, qp = 128, 64, 8, 32
        write_input(tmp_path, w, h, bits)
        r = subprocess.run([os.path.join(REF, 'EncoderAppServe')] + encoder_args(w, h, bits, qp) + ['-b', 'serve.bin'], cwd=tmp_path,
                           env=dict(env, VVCB_BROKER=path), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        assert r.returncode != 0 and 'exceeds the server' in r.stdout
    finally:
        subprocess.run([os.path.join(FAKE, 'vvcb_broker'), path, '--stop'], env=env)
        server.wait(timeout=30)


def test_frame_parallel_served_encode_gathers_to_the_sequential_bitstream(built, tmp_path):
    """The whole frame-parallel route (SURVEY.md 8e / 8f-4): one served encoder process per picture of a three-picture sequence, all sharing one
    engine context through the broker; the gather (vvc_intra_b200/assemble.py) must reproduce the bitstream the plain sequential encoder writes
    for the sequence, byte for byte."""
    from make_golden import synth_yuv
    from vvc_intra_b200 import assemble
    w, h, bits, qp, n = 64, 64, 8, 32, 3
    data = b''
    for f in range(n):
        Y, U, V = synth_yuv(w, h, bits, f)
        data += Y.tobytes() + U.tobytes() + V.tobytes()
    (tmp_path / 'in.yuv').write_bytes(data)
    (tmp_path / 'Time_python.dat').write_bytes(b'')
    args = [a for a in encoder_args(w, h, bits, qp)]
    args = args[:args.index('-f')] + args[args.index('-f') + 2:]
    path = str(tmp_path / 'broker.shm')
    envb = dict(os.environ, LD_LIBRARY_PATH=FAKE)
    server = subprocess.Popen([os.path.join(FAKE, 'vvcb_broker'), path, '--bit-depth', '8', '--clients', '4', '--frame', '64x64', '--workers', '2'],
                              env=envb, stdout=subprocess.PIPE, stderr=subprocess.STDOUT)
    try:
        seq = subprocess.Popen([os.path.join(REF, 'EncoderApp')] + args + ['-f', str(n), '-b', 'seq.bin'], cwd=tmp_path, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        procs = [subprocess.Popen([os.path.join(REF, 'EncoderAppServe')] + args + ['-f', '1', '--FrameSkip=%d' % f, '-b', 'f%d.bin' % f], cwd=tmp_path,
                                  env=dict(envb, VVCB_BROKER=path, VVCB_SHIM_REPORT=str(tmp_path / ('rep%d.json' % f))), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                 for f in range(n)]
        for p in procs:
            out, _ = p.communicate(timeout=600)
            assert p.returncode == 0, out[-3000:]
        assert seq.wait(timeout=600) == 0
        stats = json.loads(subprocess.check_output([os.path.join(FAKE, 'vvcb_broker'), path, '--stats'], env=envb))
        assert stats['clients_seen'] == n
    finally:
        subprocess.run([os.path.join(FAKE, 'vvcb_broker'), path, '--stop'], env=envb)
        try:
            server.wait(timeout=30)
        except subprocess.TimeoutExpired:
            server.kill()
    for f in range(n):
        assert json.loads((tmp_path / ('rep%d.json' % f)).read_text())['visits'] > 100
    assemble.assemble_sequential([str(tmp_path / ('f%d.bin' % f)) for f in range(n)], str(tmp_path / 'all.bin'))
    assert (tmp_path / 'all.bin').read_bytes() == (tmp_path / 'seq.bin').read_bytes()


def test_frame_parallel_driver_over_two_brokers(built, tmp_path):
    """vvc_intra_b200/frame_parallel.py: four pictures dealt over two engine contexts (two brokers -- on the GPU box two devices), at most three
    encoder processes alive at a time; bitstream and reconstruction equal the plain sequential encoder's."""
    from make_golden import synth_yuv
    from vvc_intra_b200 import frame_parallel
    w, h, bits, qp, n = 64, 64, 8, 32, 4
    data = b''
    for f in range(n):
        Y, U, V = synth_yuv(w, h, bits, f)
        data += Y.tobytes() + U.tobytes() + V.tobytes()
    (tmp_path / 'in.yuv').write_bytes(data)
    (tmp_path / 'Time_python.dat').write_bytes(b'')
    args = encoder_args(w, h, bits, qp)                                     # carries `-f 1`: the driver replaces it
    seq = subprocess.Popen([os.path.join(REF, 'EncoderApp')] + args[:args.index('-f')] + args[args.index('-f') + 2:] + ['-f', str(n), '-b', 'seq.bin', '-o', 'seq.yuv'],
                           cwd=tmp_path, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
    st = frame_parallel.encode_sequence(os.path.join(REF, 'EncoderAppServe'), args, n, str(tmp_path / 'all.bin'), devices=(0, 0), bit_depth=bits, frame_size=(w, h),
                                        workdir=str(tmp_path / 'work'), max_procs=3, broker_bin=os.path.join(FAKE, 'vvcb_broker'),
                                        env=dict(os.environ, LD_LIBRARY_PATH=FAKE), recon_path=str(tmp_path / 'all.yuv'), cwd=str(tmp_path), timeout=600)
    assert seq.wait(timeout=600) == 0
    assert (tmp_path / 'all.bin').read_bytes() == (tmp_path / 'seq.bin').read_bytes()
    assert (tmp_path / 'all.yuv').read_bytes() == (tmp_path / 'seq.yuv').read_bytes()
    assert [p['picture'] for p in st['pictures']] == [0, 1, 2, 3] and [d['pictures'] for d in st['devices']] == [2, 2]
    assert all(d['clients_seen'] == 2 and d['visits'] > 100 for d in st['devices']) and st['bytes'] == len((tmp_path / 'seq.bin').read_bytes())
    with pytest.raises(frame_parallel.FrameParallelError):                  # a failing encoder surfaces with its output
        frame_parallel.encode_sequence(os.path.join(REF, 'EncoderAppServe'), ['-c', 'missing.cfg'], 1, str(tmp_path / 'x.bin'), bit_depth=bits, frame_size=(w, h),
                                       broker_bin=os.path.join(FAKE, 'vvcb_broker'), env=dict(os.environ, LD_LIBRARY_PATH=FAKE), cwd=str(tmp_path), timeout=60)
