"""Joint Cb-Cr coding of the chroma intra candidates (vvcb_chroma_joint_tu_eval): one residual stands for Cb and Cr under TuCResMode 1..3
and CSign, is transformed, quantised (scalar or dependent, on the chroma contexts) and inverse-mapped to both reconstructions; its cbf bins,
the joint flag and the residual are priced on one carried copy of the models.

The checker is orc_chroma_joint_tu_cand in tests/chroma_joint_oracle/chroma_joint_oracle.c, composed from the functions of the chain of
vvcb_chroma_tu_eval (tests/chroma_tu_oracle/chroma_tu_oracle.c).  The forward combination is the library's restatement of JVET-O0105's
encoder derivation (H.266 does not specify it): parity unpinned.  What ties the rest down:
  - the inverse mapping equals the TuCResMode table of H.266 8.7.2 evaluated in NumPy for every r of int16;
  - with resCr = CSign * resCb, mode 2 codes exactly what vvcb_chroma_tu_eval codes for Cb;
  - the context rules: marking one model at a time moves the bits as the syntax's contexts predict;
  - the kernel source on host threads, and the device, equal the oracle chain bit for bit."""
import ctypes as C
import os
import subprocess
import sys
import time
from collections import Counter

import numpy as np
import pytest

import test_chroma_eval as CE
import test_chroma_tu_eval as TE
from test_chroma_tu_eval import QUANT, DEPQUANT, RATE, FLAG_SETS, CTU, E, _p, max_qp, model_view, uniform_states, marked_delta, MARK_STATE

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = [(m, s) for m in (1, 2, 3) for s in (1, -1)]


@pytest.fixture(scope='module')
def orc():
    """the joint chain (tests/chroma_joint_oracle); .tu: the chain of vvcb_chroma_tu_eval it links (tests/chroma_tu_oracle)"""
    subprocess.check_call(['make', '-s', '-f', 'tests/chroma_joint_oracle/Makefile'], cwd=ROOT)
    T = C.CDLL(os.path.join(ROOT, 'tests/chroma_tu_oracle/libchroma_tu_oracle.so'))
    L = C.CDLL(os.path.join(ROOT, 'tests/chroma_joint_oracle/libchroma_joint_oracle.so'))
    vp, i = C.c_void_p, C.c_int
    L.orc_chroma_joint_tu_batch.argtypes = [vp, i, vp, i, i, i, i, vp, vp, i, vp, vp, vp, vp, vp]
    T.orc_chroma_tu_batch.argtypes = [vp, i, vp, i, i, i, i, vp, vp, i, vp, vp, vp, vp, vp]
    L.orc_chroma_joint_inverse.argtypes = [vp, i, i, i, vp, vp]
    L.orc_chroma_joint_combine.argtypes = [i, i, i, i]
    L.tu = T
    return L


@pytest.fixture(scope='module')
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp('emul_chroma_joint') / 'libemul_chroma_joint.so'
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-g', '-ffp-contract=off', '-fPIC', '-shared', '-pthread', '-Wall', '-Wno-unused-function',
                           '-Wno-unknown-pragmas', '-Wno-unused-variable', '-o', str(out), os.path.join(ROOT, 'tests/host_emul/emul_chroma_joint.cpp')])
    L = C.CDLL(str(out))
    vp, i = C.c_void_p, C.c_int
    L.emul_chroma_joint_tu_eval.argtypes = [vp, i, vp, i, i, i, i, vp, i, vp, i, vp, C.c_size_t, vp, vp, vp, vp]
    return L


# ---------------------------------------------------------------------------------------------------------------------------------
# models, candidates, runs
# ---------------------------------------------------------------------------------------------------------------------------------
def random_states(rng, n):
    s = np.zeros(n, E().CHROMA_JOINT_CTX_STATES_DTYPE)
    flat = model_view(s)
    m = flat.shape[1]
    flat[:, :, 0] = rng.integers(1, 0x400, (n, m)) << 5
    flat[:, :, 1] = rng.integers(1, 0x4000, (n, m)) << 1
    flat[:, :, 2] = (rng.integers(4, 8, (n, m)) << 4) | rng.integers(4, 8, (n, m))
    return s


JOINT_FIRST = 70                                                     # Ctx::JointCbCrFlag: models 70..72 of vvcb_chroma_joint_ctx_states


def make_jobs(rng, visits, bd, per_visit=2, flags=FLAG_SETS, qps=None, n_states=8, modes=MODES):
    jobs, off, k = [], 0, 0
    for vi, v in enumerate(visits):
        n = 2 << (int(v['log2w']) + int(v['log2h']))
        cands = [c for c in range(8) if v['cclm'] or not 4 <= c <= 6]
        for t in range(per_visit):
            j = np.zeros(1, E().CHROMA_JOINT_TU_JOB_DTYPE)[0]
            j['visit'], j['cand'], j['flags'] = vi, cands[(3 * vi + 5 * t) % len(cands)], flags[k % len(flags)]
            j['mode'], j['sign'] = modes[(vi + 7 * t) % len(modes)]
            qp = int(rng.integers(12, 40)) if qps is None else qps[k % len(qps)]
            j['qp_per'], j['qp_rem'] = qp // 6, qp % 6
            j['lambda'] = 0.57 * 2 ** ((qp - 12) / 3) * 4 ** (bd - 8) * float(rng.uniform(0.7, 1.3))
            j['rate_idx'] = int(rng.integers(0, n_states))
            j['offset'] = off
            off += n
            k += 1
            jobs.append(j)
    return np.array(jobs, E().CHROMA_JOINT_TU_JOB_DTYPE), off


def _outputs(n_jobs, n_samples):
    return dict(results=np.zeros(n_jobs, E().CHROMA_JOINT_TU_RESULT_DTYPE), level=np.zeros(n_samples, np.int32),
                reco=np.zeros(n_samples, np.int16), pred=np.zeros(n_samples, np.int16))


def oracle(orc, fr, visits, jobs, states, n_samples, ctu=CTU, dep_quant=1):
    out = _outputs(len(jobs), n_samples)
    luma = np.ascontiguousarray(fr.luma)
    orc.orc_chroma_joint_tu_batch(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, dep_quant, _p(visits), _p(jobs), len(jobs),
                                  _p(states), _p(out['level']), _p(out['reco']), _p(out['pred']), _p(out['results']))
    return out


def emulate(emul, fr, visits, jobs, states, n_samples, ctu=CTU, dep_quant=1):
    out = _outputs(len(jobs), n_samples)
    luma = np.ascontiguousarray(fr.luma)
    emul.emul_chroma_joint_tu_eval(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, dep_quant, _p(visits), len(visits), _p(jobs),
                                   len(jobs), _p(states), n_samples, _p(out['level']), _p(out['reco']), _p(out['pred']), _p(out['results']))
    return out


def compare(got, want, what=''):
    for k in ('level', 'reco', 'pred'):
        if k in got:
            bad = np.flatnonzero(got[k] != want[k])
            assert not len(bad), '%s %s differs at %d samples, first %d: %d vs %d' % (what, k, len(bad), bad[0], got[k][bad[0]], want[k][bad[0]])
    r, o = got['results'], want['results']
    for f in ('abs_sum_coeff', 'abs_sum_level', 'frac_bits'):
        bad = np.flatnonzero(r['res'][f] != o['res'][f])
        assert not len(bad), '%s %s differs for job %d: %s vs %s' % (what, f, bad[0], r['res'][f][bad[0]], o['res'][f][bad[0]])
    for f in ('sse', 'cbf_bits', 'joint_bits', 'cbf'):
        bad = np.flatnonzero((r[f] != o[f]).reshape(len(r), -1).any(axis=1))
        assert not len(bad), '%s %s differs for job %d: %s vs %s' % (what, f, bad[0], r[f][bad[0]], o[f][bad[0]])
    assert r.tobytes() == o.tobytes()


def _kernel_case(rng, bd, kind):
    fr = CE.Frame(rng, bd, 160, 128, kind)
    visits = CE.make_visits(rng)
    states = random_states(rng, 8)
    qps = None if kind != 'flat' else (0, 6, max_qp(bd))
    jobs, ns = make_jobs(rng, visits, bd, per_visit=3, qps=qps)
    return fr, visits, jobs, states, ns


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
def test_struct_layout_matches_the_header(tmp_path):
    fields = {'vvcb_chroma_joint_ctx_states': ('chroma', 'joint'),
              'vvcb_chroma_joint_tu_job': ('visit', 'cand', 'flags', 'rate_idx', 'mode', 'sign', 'qp_per', 'qp_rem', 'offset', 'lambda'),
              'vvcb_chroma_joint_tu_result': ('res', 'sse', 'cbf_bits', 'joint_bits', 'cbf')}
    src = tmp_path / 'sz.c'
    body = ''.join('printf("%%zu\\n", sizeof(%s));' % s + ''.join('printf("%%zu\\n", offsetof(%s, %s));' % (s, f) for f in fs)
                   for s, fs in fields.items())
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vvc_intra_b200.h"\nint main(void){%sreturn 0;}\n' % body)
    exe = tmp_path / 'sz'
    subprocess.check_call(['gcc', '-I' + os.path.join(ROOT, 'include'), '-o', str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    eng = E()
    want = []
    for dt, fs in zip((eng.CHROMA_JOINT_CTX_STATES_DTYPE, eng.CHROMA_JOINT_TU_JOB_DTYPE, eng.CHROMA_JOINT_TU_RESULT_DTYPE), fields.values()):
        want += [dt.itemsize] + [dt.fields[f][1] for f in fs]
    assert got == want
    assert [got[0], got[3], got[14]] == [438, 32, 56]


def test_inverse_mapping_equals_the_tucresmode_table(orc):
    """H.266 8.7.2 for every r of int16, every mode and sign: computed in int (CSign * -32768 does not fit int16)"""
    r = np.arange(-32768, 32768, dtype=np.int16)
    r64 = r.astype(np.int64)
    for mode, sign in MODES:
        cb, cr = np.zeros(len(r), np.int32), np.zeros(len(r), np.int32)
        orc.orc_chroma_joint_inverse(_p(r), len(r), mode, sign, _p(cb), _p(cr))
        want = {1: (r64, (sign * r64) >> 1), 2: (r64, sign * r64), 3: ((sign * r64) >> 1, r64)}[mode]
        assert np.array_equal(cb, want[0]) and np.array_equal(cr, want[1]), (mode, sign)
    cb, cr = np.zeros(1, np.int32), np.zeros(1, np.int32)
    orc.orc_chroma_joint_inverse(_p(np.array([-32768], np.int16)), 1, 2, -1, _p(cb), _p(cr))
    assert cr[0] == 32768


def test_forward_combination_truncates_toward_zero(orc):
    f = orc.orc_chroma_joint_combine
    assert f(-7, 0, 2, 1) == -3 and f(-3, 1, 1, 1) == -2 and f(-1, 1, 1, 1) == 0 and f(1, -1, 3, 1) == 0 and f(-5, 2, 2, -1) == -3
    rng = np.random.default_rng(5)
    cb, cr = rng.integers(-1023, 1024, 4000), rng.integers(-1023, 1024, 4000)
    for mode, sign in MODES:
        num, den = {1: (4 * cb + 2 * sign * cr, 5), 2: (cb + sign * cr, 2), 3: (4 * cr + 2 * sign * cb, 5)}[mode]
        want = np.sign(num) * (np.abs(num) // den)
        got = [f(int(a), int(b), mode, sign) for a, b in zip(cb, cr)]
        assert np.array_equal(got, want), (mode, sign)


def tie_case(orc, rng, bd, sign):
    """a picture whose Cr originals are predCr + CSign * resCb inside the visits (the predictions of vvcb_chroma_eval's oracle); visits do not
    overlap, so the originals do not change any prediction"""
    fr = CE.Frame(rng, bd, 160, 128, 'noise')
    visits = np.array([CE.visit(8 + 40 * (i % 4), 8 + 40 * (i // 4), w, h, (1, w // 2, 0, h // 2, 0), dm, 1)
                       for i, (w, h, dm) in enumerate(((4, 4, 0), (8, 8, 50), (16, 8, 18), (8, 16, 1), (32, 32, 34), (16, 16, 66), (4, 16, 2),
                                                       (32, 8, 45), (8, 32, 20), (16, 32, 0), (32, 16, 50), (8, 4, 10)))], E().CHROMA_VISIT_DTYPE)
    jobs, ns = make_jobs(rng, visits, bd, per_visit=4, modes=[(2, sign)], qps=(22, 27, 32, 37))
    jobs['cand'] = jobs['cand'][::4].repeat(4)                      # one candidate per visit: its prediction is the one the originals follow
    pred = oracle(orc, fr, visits, jobs, random_states(rng, 8), ns)['pred']
    mx = (1 << bd) - 1
    for vi, v in enumerate(visits):
        j = jobs[jobs['visit'] == vi][0]
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        o = int(j['offset'])
        pcb, pcr = pred[o:o + w * h].reshape(h, w).astype(np.int64), pred[o + w * h:o + 2 * w * h].reshape(h, w).astype(np.int64)
        res = rng.integers(-(1 << (bd - 3)), 1 << (bd - 3), (h, w))
        res = np.where((pcb + res >= 0) & (pcb + res <= mx) & (pcr + sign * res >= 0) & (pcr + sign * res <= mx), res, 0)
        fr.cb[v['y']:v['y'] + h, v['x']:v['x'] + w] = pcb + res
        fr.cr[v['y']:v['y'] + h, v['x']:v['x'] + w] = pcr + sign * res
    return fr, visits, jobs, ns


def separate_twin(jobs, states):
    """the vvcb_chroma_tu_eval jobs and models that code Cb as the joint jobs code their residual"""
    tj = np.zeros(len(jobs), E().CHROMA_TU_JOB_DTYPE)
    for f in ('visit', 'cand', 'flags', 'rate_idx', 'offset'):
        tj[f] = jobs[f]
    for c in range(2):
        tj['qp_per'][:, c], tj['qp_rem'][:, c], tj['lambda'][:, c] = jobs['qp_per'], jobs['qp_rem'], jobs['lambda']
    return tj, np.ascontiguousarray(states['chroma'])


def check_tie(joint, sep, jobs, visits, bd, sign):
    mx = (1 << bd) - 1
    r, s = joint['results'], sep['results']
    assert r['cbf'].sum() > len(jobs) // 2
    inside = 0
    for i, j in enumerate(jobs):
        v = visits[j['visit']]
        n = 1 << (int(v['log2w']) + int(v['log2h']))
        o = int(j['offset'])
        assert np.array_equal(joint['level'][o:o + n], sep['level'][o:o + n]), i
        assert np.array_equal(joint['reco'][o:o + n], sep['reco'][o:o + n]), i
        assert r['sse'][i, 0] == s['comp']['sse'][i, 0] and r['res']['abs_sum_level'][i] == s['comp']['abs_sum_level'][i, 0], i
        assert r['res']['frac_bits'][i] == s['comp']['frac_bits'][i, 0], i
        assert r['cbf'][i] == s['cbf'][i, 0], i
        if r['cbf'][i]:
            assert r['cbf_bits'][i, 0] == s['cbf_bits'][i, 0], i
        pcb, pcr = joint['pred'][o:o + n].astype(np.int64), joint['pred'][o + n:o + 2 * n].astype(np.int64)
        rcb = joint['reco'][o:o + n].astype(np.int64)
        ok = (rcb > 0) & (rcb < mx)                                  # an unclipped Cb sample gives its residual r back
        assert np.array_equal(joint['reco'][o + n:o + 2 * n][ok], np.clip(pcr + sign * (rcb - pcb), 0, mx)[ok]), i
        inside += int(ok.sum())
    assert inside > 0.9 * len(joint['reco']) / 2


@pytest.mark.parametrize('sign', (1, -1))
def test_mode2_with_cr_equal_csign_cb_codes_what_the_separate_path_codes_for_cb(orc, sign):
    rng = np.random.default_rng(40 + sign)
    bd = 10
    fr, visits, jobs, ns = tie_case(orc, rng, bd, sign)
    states = random_states(rng, 8)
    joint = oracle(orc, fr, visits, jobs, states, ns)
    tj, cst = separate_twin(jobs, states)
    sep = TE.oracle(orc.tu, fr, visits, tj, cst, ns)
    check_tie(joint, sep, jobs, visits, bd, sign)


def test_emulated_kernels_context_rules(orc, emul):
    """the kernel source, every model of vvcb_chroma_joint_ctx_states marked in turn (non-adapting uniform models otherwise): the Cb cbf bin
    moves with QtCbf[Cb](0), the Cr cbf bin with QtCbf[Cr](tu_cb_coded_flag), the joint flag with JointCbCrFlag(2 * cbfCb + cbfCr - 1) and
    the residual bits as H.266's residual contexts predict on the levels it produced; all three modes, both signs"""
    rng = np.random.default_rng(21)
    St = E().CHROMA_JOINT_CTX_STATES_DTYPE
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = np.array([CE.visit(64, 40, w, h, (1, w // 2, 0, h // 2, 0), 34, 1) for w, h in CE.SHAPES], E().CHROMA_VISIT_DTYPE)
    jobs, ns = make_jobs(rng, visits, 10, per_visit=3, flags=(QUANT | RATE,), qps=(22, 27, 32), n_states=1)
    base = emulate(emul, fr, visits, jobs, uniform_states(St), ns)
    r0 = base['results']
    assert r0['cbf'].sum() > len(jobs) // 2 and {(int(m), int(s)) for m, s in zip(jobs['mode'], jobs['sign'])} == set(MODES)
    per = []
    for j in jobs:
        v = visits[j['visit']]
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        per.append(TE.chroma_residual_bins(base['level'][j['offset']:j['offset'] + w * h].reshape(h, w)))
    hit = set()
    for m in range(JOINT_FIRST + 3):
        st = uniform_states(St)
        model_view(st)[0, m, :2] = MARK_STATE
        r = emulate(emul, fr, visits, jobs, st, ns)['results']
        for i, j in enumerate(jobs):
            assert int(r['res']['frac_bits'][i]) - int(r0['res']['frac_bits'][i]) == marked_delta(per[i], m), (i, m)
            if not r0['cbf'][i]:
                assert r['cbf_bits'][i].sum() == 0 and r['joint_bits'][i] == 0
                continue
            cb, cr = int(j['mode'] != 3), int(j['mode'] != 1)
            bins = [Counter({(TE.model_index('cbf_cb', 0), cb): 1}), Counter({(TE.model_index('cbf_cr', cb), cr): 1}),
                    Counter({(JOINT_FIRST + 2 * cb + cr - 1, 1): 1})]
            got = [int(r['cbf_bits'][i, 0]) - int(r0['cbf_bits'][i, 0]), int(r['cbf_bits'][i, 1]) - int(r0['cbf_bits'][i, 1]),
                   int(r['joint_bits'][i]) - int(r0['joint_bits'][i])]
            assert got == [marked_delta(b, m) for b in bins], (i, m, int(j['mode']))
            if any(got):
                hit.add(m)
    assert {TE.model_index('cbf_cb', 0), TE.model_index('cbf_cr', 0), TE.model_index('cbf_cr', 1), 70, 71, 72} <= hit


@pytest.mark.parametrize('bd', (8, 9, 10))
@pytest.mark.parametrize('kind', ('noise', 'flat', 'checker'))
def test_emulated_kernels_match_the_oracle_chain(orc, emul, bd, kind):
    """the kernel source on host threads equals the oracle chain bit for bit: every shape 4..32, every candidate, LM on and off, modes 1..3 x
    sign +-1, the scalar and the dependent quantiser with the rate on and off; the flat picture's maximum QP codes joint residuals to zero"""
    rng = np.random.default_rng(300 + 10 * bd + len(kind))
    fr, visits, jobs, states, ns = _kernel_case(rng, bd, kind)
    assert {int(c) for c in jobs['cand']} == set(range(8)) and set(jobs['flags'].tolist()) == set(FLAG_SETS)
    assert {(int(m), int(s)) for m, s in zip(jobs['mode'], jobs['sign'])} == set(MODES)
    assert set(visits['cclm'].tolist()) == {0, 1}
    want = oracle(orc, fr, visits, jobs, states, ns)
    got = emulate(emul, fr, visits, jobs, states, ns)
    compare(got, want, '%d-bit %s' % (bd, kind))
    res = want['results']
    assert res['cbf'].any() and (res['res']['frac_bits'] > 0).any() and (res['joint_bits'] > 0).any()
    if kind == 'flat':
        zero = res['cbf'] == 0
        assert zero.any() and (res['cbf_bits'][zero] == 0).all() and (res['joint_bits'][zero] == 0).all()


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def run_device(fr, visits, jobs, states, ns, ctu=CTU):
    with CE._engine(fr, ctu) as eng:
        return eng.chroma_joint_tu_eval(visits, jobs, ns, states=states, want_level=True, want_reco=True, want_pred=True)


@pytest.mark.gpu
@pytest.mark.parametrize('bd', (8, 9, 10))
def test_device_matches_oracle_chain(orc, bd):
    """mixed batches and walk-sized ones (30 CUs x the three modes, dependent quantiser + rate) on noise and checker pictures"""
    rng = np.random.default_rng(400 + bd)
    for kind in ('noise', 'checker', 'flat'):
        fr, visits, jobs, states, ns = _kernel_case(rng, bd, kind)
        compare(run_device(fr, visits, jobs, states, ns), oracle(orc, fr, visits, jobs, states, ns), '%d-bit %s' % (bd, kind))
        walk = visits[rng.permutation(len(visits))[:30]]
        wj, wns = make_jobs(rng, walk, bd, per_visit=3, flags=(QUANT | DEPQUANT | RATE,), modes=[(1, 1), (2, -1), (3, 1)])
        compare(run_device(fr, walk, wj, states, wns), oracle(orc, fr, walk, wj, states, wns), 'walk %d-bit %s' % (bd, kind))


@pytest.mark.gpu
def test_device_batch_above_one_chunk(orc):
    """more than 65 536 candidates: two chunks of the internal 16-bit rate index"""
    rng = np.random.default_rng(500)
    fr, visits, jobs, states, ns = _kernel_case(rng, 10, 'noise')
    want = oracle(orc, fr, visits, jobs, states, ns)
    reps = -(-70000 // len(jobs))
    big = np.tile(jobs, reps)
    big['offset'] += np.repeat(np.arange(reps, dtype=np.uint32) * ns, len(jobs))
    with CE._engine(fr) as eng:
        got = eng.chroma_joint_tu_eval(visits, big, ns * reps, states=states, want_level=True, want_reco=True)
    assert len(big) > 65536
    assert got['results'].tobytes() == np.tile(want['results'], reps).tobytes()
    assert np.array_equal(got['level'], np.tile(want['level'], reps)) and np.array_equal(got['reco'], np.tile(want['reco'], reps))


@pytest.mark.gpu
@pytest.mark.parametrize('bd', (8, 9, 10))
def test_device_extreme_qps_with_saturated_residuals(orc, bd):
    """chroma QP 0 and the maximum for the bit depth on pictures whose residuals reach +(2^bd - 1) in Cb and -(2^bd - 1) in Cr: mode 2 with
    CSign = -1 codes a full-scale residual whose inverse mapping drives both reconstructions into their clips"""
    rng = np.random.default_rng(600 + bd)
    mx = (1 << bd) - 1
    fr = CE.Frame(rng, bd, 160, 128, 'noise')
    fr.cb[:], fr.cb_reco[:], fr.cr[:], fr.cr_reco[:], fr.luma[:] = mx, 0, 0, mx, 0
    visits = CE.make_visits(rng)
    states = random_states(rng, 8)
    jobs, ns = make_jobs(rng, visits, bd, per_visit=3, qps=(0, max_qp(bd)), modes=[(2, -1), (1, 1), (2, -1), (3, -1)])
    want = oracle(orc, fr, visits, jobs, states, ns)
    compare(run_device(fr, visits, jobs, states, ns), want, '%d-bit extreme QP' % bd)
    hits = 0
    for j in jobs[(jobs['mode'] == 2) & (jobs['sign'] == -1) & (jobs['qp_per'] == 0)]:
        v = visits[j['visit']]
        n = 1 << (int(v['log2w']) + int(v['log2h']))
        o = int(j['offset'])
        lv = want['level'][o:o + n]
        hits += int(np.abs(lv).max() > 0 and (want['reco'][o:o + n] == mx).any() and (want['reco'][o + n:o + 2 * n] == 0).any())
    assert hits > 10


@pytest.mark.gpu
def test_device_predictions_and_the_mode2_tie(orc):
    """the device's predictions equal vvcb_chroma_eval's; with resCr = CSign * resCb, mode 2 equals vvcb_chroma_tu_eval's Cb on the device"""
    rng = np.random.default_rng(700)
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = CE.make_visits(rng)
    jobs, ns = make_jobs(rng, visits, 10, per_visit=8, flags=(QUANT,))
    with CE._engine(fr) as eng:
        _, blocks = eng.chroma_eval(visits, want_pred=True)
        got = eng.chroma_joint_tu_eval(visits, jobs, ns, want_pred=True)
    for j in jobs:
        b = blocks[j['visit']][j['cand']]
        assert np.array_equal(got['pred'][j['offset']:j['offset'] + b.size], b.ravel())
    for sign in (1, -1):
        fr, visits, jobs, ns = tie_case(orc, rng, 10, sign)
        states = random_states(rng, 8)
        tj, cst = separate_twin(jobs, states)
        with CE._engine(fr) as eng:
            joint = eng.chroma_joint_tu_eval(visits, jobs, ns, states=states, want_level=True, want_reco=True, want_pred=True)
            sep = eng.chroma_tu_eval(visits, tj, ns, states=cst, want_level=True, want_reco=True, want_pred=True)
        check_tie(joint, sep, jobs, visits, 10, sign)


@pytest.mark.gpu
def test_refusals(tmp_path):
    """every refusal returns its code and error string and leaves the context usable; the broker proxy refuses the entry point"""
    import vvc_intra_b200 as vb
    eng_mod = E()
    rng = np.random.default_rng(9)
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = np.array([CE.visit(64, 40, 8, 8, (1, 4, 4, 4, 4), 5, 1), CE.visit(64, 64, 8, 8, (1, 4, 4, 4, 4), 5, 0)], eng_mod.CHROMA_VISIT_DTYPE)
    states = random_states(rng, 2)
    jobs, ns = make_jobs(rng, visits[:1], 10, per_visit=1, flags=(QUANT | DEPQUANT | RATE,), n_states=2)
    good = jobs[0]

    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=CTU) as eng:
        eng.frame_begin(np.zeros((256, 320), np.int16))
        last = lambda: eng._lib.vvcb_last_error(eng._ctx).decode()
        rc = eng._lib.vvcb_chroma_joint_tu_eval(eng._ctx, _p(visits), 2, _p(jobs), 1, _p(states), 2, ns, None, None, None,
                                                _p(np.zeros(1, eng_mod.CHROMA_JOINT_TU_RESULT_DTYPE)))
        assert rc == -3 and 'vvcb_chroma_frame_begin has not been called' in last()
        eng.reco_update(fr.luma)
        eng.chroma_frame_begin(fr.cb, fr.cr)
        ref = eng.chroma_joint_tu_eval(visits, jobs, ns, states=states)['results']

        def call(v, j, st=states, n=ns):
            out = np.zeros(len(j), eng_mod.CHROMA_JOINT_TU_RESULT_DTYPE)
            return eng._lib.vvcb_chroma_joint_tu_eval(eng._ctx, _p(v), len(v), _p(j), len(j), _p(st) if st is not None else None,
                                                      0 if st is None else len(st), n, None, None, None, _p(out))
        cases = []
        for f, val, why in (('visit', 2, 'visit index out of range'), ('cand', 8, 'cand above 7'), ('flags', 0, 'flags'),
                            ('flags', QUANT | 4, 'flags'), ('flags', QUANT | 8, 'flags'), ('flags', QUANT | 64, 'flags'),
                            ('rate_idx', 2, 'rate_idx'), ('offset', ns - 1, 'outside n_samples'), ('mode', 0, 'mode'), ('mode', 4, 'mode'),
                            ('sign', 0, 'sign'), ('sign', 2, 'sign'), ('sign', -2, 'sign'), ('lambda', 0.0, 'lambda'), ('lambda', -1.0, 'lambda'),
                            ('lambda', float('inf'), 'lambda'), ('lambda', float('nan'), 'lambda')):
            b = good.copy()
            b[f] = val
            cases.append((b, why))
        for per, rem in ((-1, 0), (0, -1), (0, 6), (max_qp(10) // 6, max_qp(10) % 6 + 1), (13, 0)):
            b = good.copy()
            b['qp_per'], b['qp_rem'] = per, rem
            cases.append((b, 'qp_per / qp_rem out of range'))
        lm_off = good.copy()
        lm_off['visit'], lm_off['cand'] = 1, 5
        cases.append((lm_off, 'LM candidate of a visit without cclm'))
        for b, why in cases:
            assert call(visits, np.array([good, b])) == -1, b
            assert last().startswith('vvcb_chroma_joint_tu_eval: job 1: ') and why in last(), (why, last())
        assert call(visits, np.array([good]), st=None) == -1 and 'rate_idx' in last()
        bv = visits.copy()
        bv[1]['log2w'] = 6
        assert call(bv, np.array([good])) == -1 and last().startswith('vvcb_chroma_joint_tu_eval: visit 1: ')
        dq_free = good.copy()
        dq_free['flags'], dq_free['lambda'] = QUANT, 0.0
        assert call(visits, np.array([dq_free]), st=None) == 0
        assert eng.chroma_joint_tu_eval(visits, jobs, ns, states=states)['results'].tobytes() == ref.tobytes()
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([os.path.join(ROOT, 'vvc_intra_b200/vvcb_broker'), path, '--bit-depth', '10', '--ctu', str(CTU), '--clients', '2',
                               '--frame', '320x256', '--workers', '1'], env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        prog = ('import numpy as np, vvc_intra_b200 as vb\n'
                'from vvc_intra_b200 import engine as E\n'
                'eng = vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=%d)\n'
                'eng.frame_begin(np.zeros((256, 320), np.int16))\n'
                'j = np.zeros(1, E.CHROMA_JOINT_TU_JOB_DTYPE); j["flags"] = 1; j["mode"] = 2; j["sign"] = 1\n'
                'try:\n'
                '    eng.chroma_joint_tu_eval(np.zeros(1, E.CHROMA_VISIT_DTYPE), j, 64); print("accepted")\n'
                'except E.EngineError as e:\n'
                '    print("broker" in str(e))\n') % CTU
        r = None
        for _ in range(100):
            if os.path.exists(path):
                r = subprocess.run([sys.executable, '-c', prog], cwd=ROOT, env=dict(env0, VVCB_BROKER=path), stdout=subprocess.PIPE,
                                   stderr=subprocess.STDOUT, text=True, timeout=300)
                break
            time.sleep(0.2)
        assert r is not None and r.returncode == 0, r and r.stdout[-2000:]
        assert r.stdout.strip().splitlines()[-1] == 'True', r.stdout[-2000:]
    finally:
        subprocess.run([os.path.join(ROOT, 'vvc_intra_b200/vvcb_broker'), path, '--stop'], env=env0, timeout=60)
        try:
            server.wait(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()


@pytest.mark.gpu
def test_alternating_with_the_separate_call_equals_fresh_contexts():
    """one context alternates vvcb_chroma_tu_eval and vvcb_chroma_joint_tu_eval with growing, then shrinking batches (they share the staging
    slots): every output equals the same call on a fresh context, byte for byte"""
    rng = np.random.default_rng(900)
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = CE.make_visits(rng)
    calls = []
    for per in (1, 4, 12, 3, 1):
        tj, tns = TE.make_jobs(rng, visits, 10, per_visit=per)
        jj, jns = make_jobs(rng, visits, 10, per_visit=per)
        ts, js = TE.random_states(rng, 8), random_states(rng, 8)
        calls.append(lambda eng, tj=tj, tns=tns, ts=ts: eng.chroma_tu_eval(visits, tj, tns, states=ts, want_level=True, want_reco=True, want_pred=True))
        calls.append(lambda eng, jj=jj, jns=jns, js=js: eng.chroma_joint_tu_eval(visits, jj, jns, states=js, want_level=True, want_reco=True,
                                                                                  want_pred=True))
    with CE._engine(fr) as eng:
        shared = [c(eng) for c in calls]
    for c, got in zip(calls, shared):
        with CE._engine(fr) as eng:
            want = c(eng)
        assert all(got[k].tobytes() == want[k].tobytes() for k in want)
