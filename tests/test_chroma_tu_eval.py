"""Chroma TU coding of the chroma intra candidates (vvcb_chroma_tu_eval): Cb and Cr transformed, quantised (scalar or dependent, on the chroma
contexts), reconstructed and priced (cbf bins, residual bits) on one carried copy of the models.

The checker is the plain-C chain of tests/chroma_tu_oracle/chroma_tu_oracle.c: the chroma prediction of oracle/vvc_oracle_chroma.c and the
oracle's transform, quantisers and rate estimation, whose dependent quantiser and residual rate run the pinned luma code with the chroma
context derivations of H.266 substituted (tests/chroma_tu_oracle/Makefile).  Nothing here compares with the reference encoder's own chroma coding.
What ties it down:
  - the context indices: with every model identical and non-adapting but one, the bits move by exactly what a direct Python evaluation of the
    H.266 derivations (9.3.4.2.4-9.3.4.2.8) predicts, for every model, in the oracle and in the kernel source;
  - context-blind equivalence with the pinned luma path: with all models identical and non-adapting the chroma quantiser and rate equal the
    luma ones (oracle here, device against vvcb_tu_eval on the GPU);
  - the kernel source on host threads, and the device, equal the oracle chain bit for bit."""
import ctypes as C
import os
import re
import subprocess
import sys
import time
from collections import Counter

import numpy as np
import pytest

import test_chroma_eval as CE                  # the chroma picture, visit and availability helpers of the prediction stage

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
QUANT, DEPQUANT, RATE = 1, 2, 32
FLAG_SETS = (QUANT, QUANT | RATE, QUANT | DEPQUANT, QUANT | DEPQUANT | RATE)
CTU = CE.CTU


def E():
    import vvc_intra_b200.engine as eng
    return eng


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def max_qp(bd):
    return 63 + 6 * (bd - 8)


@pytest.fixture(scope='module')
def orc():
    subprocess.check_call(['make', '-s', '-f', 'tests/chroma_tu_oracle/Makefile'], cwd=ROOT)
    L = C.CDLL(os.path.join(ROOT, 'tests/chroma_tu_oracle/libchroma_tu_oracle.so'))
    vp, i = C.c_void_p, C.c_int
    L.orc_chroma_tu_batch.argtypes = [vp, i, vp, i, i, i, i, vp, vp, i, vp, vp, vp, vp, vp]
    L.orc_chroma_residual_bits.argtypes = [vp, i, i, i, vp]
    L.orc_chroma_residual_bits.restype = C.c_uint64
    L.orc_residual_bits.argtypes = [vp, i, i, i, i, i, i, vp]
    L.orc_residual_bits.restype = C.c_uint64
    for f in (L.orc_dep_quant, L.orc_dep_quant_chroma):
        f.argtypes = [vp, i, i, i, i, i, i, C.c_double, vp, i, vp]
    L.orc_fwd_transform.argtypes = [vp, i, i, i, i, i, vp]
    return L


@pytest.fixture(scope='module')
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp('emul_chroma_tu') / 'libemul_chroma.so'
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-g', '-ffp-contract=off', '-fPIC', '-shared', '-pthread', '-Wall', '-Wno-unused-function',
                           '-Wno-unknown-pragmas', '-Wno-unused-variable', '-o', str(out), os.path.join(ROOT, 'tests/host_emul/emul_chroma_tu.cpp')])
    L = C.CDLL(str(out))
    vp, i = C.c_void_p, C.c_int
    L.emul_chroma_tu_eval.argtypes = [vp, i, vp, i, i, i, i, vp, i, vp, i, vp, C.c_size_t, vp, vp, vp, vp]
    return L


def frac_bits_table():
    src = open(os.path.join(ROOT, 'vvc_intra_b200/csrc/vvc_rom_tables.h')).read()
    body = re.search(r'kBinFracBits\[512\] = \{(.*?)\};', src, re.S).group(1)
    t = [int(x) for x in re.findall(r'\d+', body)]
    assert len(t) == 512
    return t


FB = frac_bits_table()


# ---------------------------------------------------------------------------------------------------------------------------------
# models, candidates, runs
# ---------------------------------------------------------------------------------------------------------------------------------
def model_view(s):
    """per model: state0, state1, rate | pad << 8"""
    return s.view(np.uint8).reshape(len(s), -1).view(np.uint16).reshape(len(s), -1, 3)


def random_states(rng, n):
    s = np.zeros(n, E().CHROMA_CTX_STATES_DTYPE)
    flat = model_view(s)
    m = flat.shape[1]
    flat[:, :, 0] = rng.integers(1, 0x400, (n, m)) << 5
    flat[:, :, 1] = rng.integers(1, 0x4000, (n, m)) << 1
    flat[:, :, 2] = (rng.integers(4, 8, (n, m)) << 4) | rng.integers(4, 8, (n, m))
    return s


BASE_STATE, MARK_STATE = (16384, 16384), (4096, 4096)        # window rates 15 / 15: BinProbModel_Std::update leaves the state unchanged


def uniform_states(dtype, n=1, state=BASE_STATE):
    s = np.zeros(n, dtype)
    flat = model_view(s)
    flat[:, :, 0], flat[:, :, 1], flat[:, :, 2] = state[0], state[1], 0xff
    return s


def model_index(field, *idx):
    """flat position of a chroma model in vvcb_chroma_ctx_states"""
    dt = E().CHROMA_CTX_STATES_DTYPE
    sub = dt.fields[field][0]
    shape = sub.shape
    return dt.fields[field][1] // 6 + (int(np.ravel_multi_index(idx, shape)) if shape else 0)


def make_jobs(rng, visits, bd, per_visit=2, flags=FLAG_SETS, qps=None, n_states=8):
    jobs, off, k = [], 0, 0
    for vi, v in enumerate(visits):
        n = 2 << (int(v['log2w']) + int(v['log2h']))
        cands = [c for c in range(8) if v['cclm'] or not 4 <= c <= 6]
        for t in range(per_visit):
            j = np.zeros(1, E().CHROMA_TU_JOB_DTYPE)[0]
            j['visit'], j['cand'], j['flags'] = vi, cands[(3 * vi + 5 * t) % len(cands)], flags[k % len(flags)]
            for c in range(2):
                qp = int(rng.integers(12, 40)) if qps is None else qps[k % len(qps)]
                j['qp_per'][c], j['qp_rem'][c] = qp // 6, qp % 6
                j['lambda'][c] = 0.57 * 2 ** ((qp - 12) / 3) * 4 ** (bd - 8) * float(rng.uniform(0.7, 1.3))
            j['rate_idx'] = int(rng.integers(0, n_states))
            j['offset'] = off
            off += n
            k += 1
            jobs.append(j)
    return np.array(jobs, E().CHROMA_TU_JOB_DTYPE), off


def oracle(orc, fr, visits, jobs, states, n_samples, ctu=CTU, dep_quant=1):
    out = dict(results=np.zeros(len(jobs), E().CHROMA_TU_RESULT_DTYPE), level=np.zeros(n_samples, np.int32),
               reco=np.zeros(n_samples, np.int16), pred=np.zeros(n_samples, np.int16))
    luma = np.ascontiguousarray(fr.luma)
    orc.orc_chroma_tu_batch(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, dep_quant, _p(visits), _p(jobs), len(jobs), _p(states),
                            _p(out['level']), _p(out['reco']), _p(out['pred']), _p(out['results']))
    return out


def emulate(emul, fr, visits, jobs, states, n_samples, ctu=CTU, dep_quant=1):
    out = dict(results=np.zeros(len(jobs), E().CHROMA_TU_RESULT_DTYPE), level=np.zeros(n_samples, np.int32),
               reco=np.zeros(n_samples, np.int16), pred=np.zeros(n_samples, np.int16))
    luma = np.ascontiguousarray(fr.luma)
    emul.emul_chroma_tu_eval(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, dep_quant, _p(visits), len(visits), _p(jobs), len(jobs),
                             _p(states), n_samples, _p(out['level']), _p(out['reco']), _p(out['pred']), _p(out['results']))
    return out


def compare(got, want, what=''):
    for k in ('level', 'reco', 'pred'):
        if k in got:
            bad = np.flatnonzero(got[k] != want[k])
            assert not len(bad), '%s %s differs at %d samples, first %d: %d vs %d' % (what, k, len(bad), bad[0], got[k][bad[0]], want[k][bad[0]])
    r, o = got['results'], want['results']
    for f in ('abs_sum_coeff', 'abs_sum_level', 'sse', 'frac_bits'):
        bad = np.flatnonzero((r['comp'][f] != o['comp'][f]).any(axis=1))
        assert not len(bad), '%s %s differs for job %d: %s vs %s' % (what, f, bad[0], r['comp'][f][bad[0]], o['comp'][f][bad[0]])
    for f in ('cbf', 'cbf_bits'):
        bad = np.flatnonzero((r[f] != o[f]).any(axis=1))
        assert not len(bad), '%s %s differs for job %d: %s vs %s' % (what, f, bad[0], r[f][bad[0]], o[f][bad[0]])
    assert r.tobytes() == o.tobytes()


# ---------------------------------------------------------------------------------------------------------------------------------
# H.266 9.3.4.2.4-9.3.4.2.8 and 7.3.10.11, chroma, evaluated directly: the context-coded bins residual_coding spends on given levels
# ---------------------------------------------------------------------------------------------------------------------------------
GROUP_IDX = [0, 1, 2, 3, 4, 4, 5, 5, 6, 6, 6, 6, 7, 7, 7, 7] + [8] * 8 + [9] * 8


def diag_scan(bw, bh):
    return [(d - y, y) for d in range(bw + bh - 1) for y in range(min(d, bh - 1), max(0, d - bw + 1) - 1, -1)]


def chroma_residual_bins(lv, dep_quant=1):
    """Counter {(flat model index, bin): count} of the context-coded bins of residual_coding for a chroma block of levels lv (h x w)"""
    h, w = lv.shape
    sbs = diag_scan(w // 4, h // 4)
    pos = [(4 * sx + x, 4 * sy + y) for sx, sy in sbs for x, y in diag_scan(4, 4)]
    nz = [i for i, (x, y) in enumerate(pos) if lv[y, x]]
    bins = Counter()
    if not nz:
        return bins
    last = nz[-1]
    lx, ly = pos[last]
    for g, size, field in ((GROUP_IDX[lx], w, 'last_x'), (GROUP_IDX[ly], h, 'last_y')):
        shift = min(2, max(0, size >> 3))                         # ctxOffset 20 (the chroma contexts), ctxShift Clip3(0, 2, size >> 3)
        for k in range(g):
            bins[(model_index(field, k >> shift), 1)] += 1
        if g < GROUP_IDX[size - 1]:
            bins[(model_index(field, g >> shift), 0)] += 1
    a = np.abs(lv.astype(np.int64))

    def tmpl(x, y):
        s1 = npos = 0
        for dx, dy in ((1, 0), (2, 0), (0, 1), (0, 2), (1, 1)):
            if x + dx < w and y + dy < h:
                v = int(a[y + dy, x + dx])
                s1 += min(4 + (v & 1), v)
                npos += v != 0
        return s1, npos
    state, rem_bins = 0, (w * h * 7) >> 2
    coded = set()
    for sb in range(last >> 4, -1, -1):
        sx, sy = sbs[sb]
        sig = any(a[4 * sy + y, 4 * sx + x] for x, y in diag_scan(4, 4))
        if sig:
            coded.add((sx, sy))
        is_last = sb == last >> 4
        if not is_last and sb:
            ctx = int((sx + 1, sy) in coded or (sx, sy + 1) in coded)   # coded_sub_block_flag: csbfCtx + 2 (the chroma pair)
            bins[(model_index('sig_sbb', ctx), int(sig))] += 1
            if not sig:
                continue
        first = last if is_last else 16 * sb + 15
        infer = first if is_last else (16 * sb if sb else -1)
        n_nz = 0
        n = first
        while n >= 16 * sb and rem_bins >= 4:
            x, y = pos[n]
            v = int(a[y, x])
            s1, npos = tmpl(x, y)
            d = x + y
            if n_nz or n != infer:
                # sig_coeff_flag: ctxInc 36 + 8 * max(0, QState - 1) + (d < 2 ? 4 : 0) + min((locSumAbsPass1 + 1) >> 1, 3)
                bins[(model_index('sig', max(0, state - 1), (4 if d < 2 else 0) + min((s1 + 1) >> 1, 3)), int(v != 0))] += 1
                rem_bins -= 1
            if v:
                # abs_level_gtx_flag[0] / par_level_flag / abs_level_gtx_flag[1]: 0 at the last position, else 1 + (d == 0 ? 5 : 0) + min(s1 - numSig, 4)
                off = 0 if n == last else 1 + (5 if d == 0 else 0) + min(s1 - npos, 4)
                n_nz += 1
                bins[(model_index('gt1', off), int(v > 1))] += 1
                rem_bins -= 1
                if v > 1:
                    bins[(model_index('par', off), (v - 2) & 1)] += 1
                    bins[(model_index('gt2', off), int(v > 3))] += 1
                    rem_bins -= 2
            if dep_quant:
                state = (32040 >> ((state << 2) + ((v & 1) << 1))) & 3
            n -= 1
        while n >= 16 * sb:                                           # bypass-coded positions: the state machine goes on
            x, y = pos[n]
            if dep_quant:
                state = (32040 >> ((state << 2) + ((int(a[y, x]) & 1) << 1))) & 3
            n -= 1
    return bins


def marked_delta(bins, m):
    q0, q1 = (BASE_STATE[0] + BASE_STATE[1]) >> 8, (MARK_STATE[0] + MARK_STATE[1]) >> 8
    return sum(c * (FB[2 * q1 + b] - FB[2 * q0 + b]) for (mi, b), c in bins.items() if mi == m)


def level_blocks(rng, w, h, k=3):
    """quantiser-like levels: dense and large near DC, sparse towards high frequencies, one block with a lone level"""
    out = []
    yy, xx = np.mgrid[0:h, 0:w]
    for i in range(k):
        p = np.exp(-(xx + yy) / (2.0 + 3 * i))
        mag = rng.geometric(0.35 - 0.1 * i, (h, w)) * (rng.random((h, w)) < p)
        lv = (mag * rng.choice((-1, 1), (h, w))).astype(np.int32)
        out.append(lv)
    lone = np.zeros((h, w), np.int32)
    lone[int(rng.integers(0, h)), int(rng.integers(0, w))] = 1
    out.append(lone)
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
def test_struct_sizes_match_the_header(tmp_path):
    src = tmp_path / 'sz.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vvc_intra_b200.h"\n'
                   'int main(void){printf("%zu %zu %zu %zu %zu %zu %zu %zu %zu %zu\\n", sizeof(vvcb_chroma_ctx_states), sizeof(vvcb_chroma_tu_job), '
                   'sizeof(vvcb_chroma_tu_result), offsetof(vvcb_chroma_ctx_states, sig_sbb), offsetof(vvcb_chroma_ctx_states, last_y), '
                   'offsetof(vvcb_chroma_tu_job, qp_per), offsetof(vvcb_chroma_tu_job, offset), offsetof(vvcb_chroma_tu_job, lambda), '
                   'offsetof(vvcb_chroma_tu_result, cbf_bits), offsetof(vvcb_chroma_tu_result, cbf));return 0;}\n')
    exe = tmp_path / 'sz'
    subprocess.check_call(['gcc', '-I' + os.path.join(ROOT, 'include'), '-o', str(exe), str(src)])
    got = [int(x) for x in subprocess.check_output([str(exe)]).split()]
    eng = E()
    S, J, R = eng.CHROMA_CTX_STATES_DTYPE, eng.CHROMA_TU_JOB_DTYPE, eng.CHROMA_TU_RESULT_DTYPE
    assert got == [S.itemsize, J.itemsize, R.itemsize, S.fields['sig_sbb'][1], S.fields['last_y'][1], J.fields['qp_per'][1],
                   J.fields['offset'][1], J.fields['lambda'][1], R.fields['cbf_bits'][1], R.fields['cbf'][1]]
    assert got[:3] == [420, 40, 64]


def test_context_indices_of_the_oracle_equal_the_h266_derivations(orc):
    """every chroma shape, every residual context: marking that one context moves the oracle's bits by exactly what the Python evaluation of
    the H.266 derivations predicts (which also pins which positions use it), with and without the dependent quantiser's state machine"""
    rng = np.random.default_rng(11)
    St = E().CHROMA_CTX_STATES_DTYPE
    first = model_index('sig_sbb', 0)
    hit = set()
    for w, h in CE.SHAPES:
        for lv in level_blocks(rng, w, h):
            lv = np.ascontiguousarray(lv)
            for dq in (0, 1):
                bins = chroma_residual_bins(lv, dq)
                base = uniform_states(St)
                b0 = orc.orc_chroma_residual_bits(_p(lv), w, h, dq, _p(base))
                for m in range(first, 70):
                    st = uniform_states(St)
                    model_view(st)[0, m, :2] = MARK_STATE
                    got = orc.orc_chroma_residual_bits(_p(lv), w, h, dq, _p(st)) - b0
                    assert got == marked_delta(bins, m), (w, h, dq, m)
                    if got:
                        hit.add(m)
    assert hit == set(range(first, 70)), sorted(set(range(first, 70)) - hit)   # every residual context was reached


def test_context_blind_quantiser_and_rate_equal_the_pinned_luma_path(orc):
    """all models identical and non-adapting: the chroma dependent quantiser equals orc_dep_quant and the chroma residual bits equal
    orc_residual_bits (both pinned to reference records) on the same input"""
    eng = E()
    rng = np.random.default_rng(12)
    rates = np.zeros(1, eng.DQ_RATES_DTYPE)
    q = (20000 + 9000) >> 8
    rv = rates.view(np.uint32).reshape(-1, 2)
    rv[:, 0], rv[:, 1] = FB[2 * q], FB[2 * q + 1]
    lst = uniform_states(eng.CTX_STATES_DTYPE, state=(20000, 9000))
    cst = uniform_states(eng.CHROMA_CTX_STATES_DTYPE, state=(20000, 9000))
    n = 0
    for bd in (8, 10):
        for w, h in CE.SHAPES:
            for qp in (4, 22, 37, max_qp(bd)):
                resi = np.ascontiguousarray(rng.integers(-(1 << bd) + 1, 1 << bd, (h, w)) >> int(rng.integers(0, bd)), np.int16)
                coeff = np.zeros((h, w), np.int32)
                orc.orc_fwd_transform(_p(resi), w, w, h, bd, 0, _p(coeff))
                lam = 0.57 * 2 ** ((qp - 12) / 3) * 4 ** (bd - 8)
                delta = int(rng.integers(-20000, 20000))
                a, b = np.zeros((h, w), np.int32), np.zeros((h, w), np.int32)
                sa = orc.orc_dep_quant(_p(coeff), w, h, bd, 0, 0, qp, lam, _p(rates), delta, _p(a))
                sb = orc.orc_dep_quant_chroma(_p(coeff), w, h, bd, 0, 0, qp, lam, _p(rates), delta, _p(b))
                assert sa == sb and np.array_equal(a, b), (bd, w, h, qp)
                for dq in (0, 1):
                    lb = orc.orc_residual_bits(_p(a), w, h, 0, 0, 0, dq, _p(lst))
                    cb = orc.orc_chroma_residual_bits(_p(a), w, h, dq, _p(cst.copy()))
                    assert lb == cb, (bd, w, h, qp, dq)
                n += sa != 0
    assert n > 48                                                     # about half the cases keep levels


def _kernel_case(rng, bd, kind):
    fr = CE.Frame(rng, bd, 160, 128, kind)
    visits = CE.make_visits(rng)
    states = random_states(rng, 8)
    qps = None if kind != 'flat' else (0, 6, max_qp(bd))
    jobs, ns = make_jobs(rng, visits, bd, per_visit=2, qps=qps)
    return fr, visits, jobs, states, ns


@pytest.mark.parametrize('bd', (8, 9, 10))
@pytest.mark.parametrize('kind', ('noise', 'flat', 'checker'))
def test_emulated_kernels_match_the_oracle_chain(orc, emul, bd, kind):
    """the kernel source on host threads equals the oracle chain bit for bit: every shape 4..32, every candidate, LM on and off, the
    availability crossings of the prediction tests, the scalar and the dependent quantiser with the rate on and off"""
    rng = np.random.default_rng(300 + 10 * bd + len(kind))
    fr, visits, jobs, states, ns = _kernel_case(rng, bd, kind)
    assert {int(c) for c in jobs['cand']} == set(range(8)) and set(jobs['flags'].tolist()) == set(FLAG_SETS)
    want = oracle(orc, fr, visits, jobs, states, ns)
    got = emulate(emul, fr, visits, jobs, states, ns)
    compare(got, want, '%d-bit %s' % (bd, kind))
    res = want['results']
    assert res['cbf'].any() and (res['comp']['frac_bits'] > 0).any()
    if kind == 'flat':
        assert (res['cbf'] == 0).any()                                # the maximum QP codes no level


def test_emulated_kernels_context_indices(orc, emul):
    """the kernel source: marking one model at a time (non-adapting uniform models otherwise) moves the Cb / Cr residual bits and the cbf bits
    by exactly the H.266 prediction on the levels it produced"""
    rng = np.random.default_rng(21)
    St = E().CHROMA_CTX_STATES_DTYPE
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = np.array([CE.visit(64, 40, w, h, (1, w // 2, 0, h // 2, 0), 34, 1) for w, h in CE.SHAPES], E().CHROMA_VISIT_DTYPE)
    jobs, ns = make_jobs(rng, visits, 10, per_visit=2, flags=(QUANT | RATE,), qps=(27, 32, 22, 40), n_states=1)
    base = emulate(emul, fr, visits, jobs, uniform_states(St), ns)
    per = []
    for i, j in enumerate(jobs):
        v = visits[j['visit']]
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        lv = base['level'][j['offset']:j['offset'] + 2 * w * h].reshape(2, h, w)
        per.append([chroma_residual_bins(lv[0]), chroma_residual_bins(lv[1])])
    r0 = base['results']
    assert r0['cbf'].all(axis=1).sum() > len(jobs) // 2
    for m in range(70):
        st = uniform_states(St)
        model_view(st)[0, m, :2] = MARK_STATE
        r = emulate(emul, fr, visits, jobs, st, ns)['results']
        for i in range(len(jobs)):
            cbf = r0['cbf'][i]
            for c in range(2):
                assert int(r['comp']['frac_bits'][i, c]) - int(r0['comp']['frac_bits'][i, c]) == marked_delta(per[i][c], m), (i, c, m)
            cbins = [Counter({(model_index('cbf_cb', 0), int(cbf[0])): 1}), Counter({(model_index('cbf_cr', int(cbf[0])), int(cbf[1])): 1})]
            for c in range(2):
                assert int(r['cbf_bits'][i, c]) - int(r0['cbf_bits'][i, c]) == marked_delta(cbins[c], m), (i, c, m)


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def run_device(fr, visits, jobs, states, ns, ctu=CTU):
    with CE._engine(fr, ctu) as eng:
        return eng.chroma_tu_eval(visits, jobs, ns, states=states, want_level=True, want_reco=True, want_pred=True)


@pytest.mark.gpu
@pytest.mark.parametrize('bd', (8, 9, 10))
def test_device_matches_oracle_chain(orc, bd):
    """walk-sized (30 CUs x 3 candidates, dependent quantiser + rate) and mixed batches on noise and checker pictures"""
    rng = np.random.default_rng(400 + bd)
    for kind in ('noise', 'checker'):
        fr, visits, jobs, states, ns = _kernel_case(rng, bd, kind)
        compare(run_device(fr, visits, jobs, states, ns), oracle(orc, fr, visits, jobs, states, ns), '%d-bit %s' % (bd, kind))
        walk = visits[rng.permutation(len(visits))[:30]]
        wj, wns = make_jobs(rng, walk, bd, per_visit=3, flags=(QUANT | DEPQUANT | RATE,))
        compare(run_device(fr, walk, wj, states, wns), oracle(orc, fr, walk, wj, states, wns), 'walk %d-bit %s' % (bd, kind))


@pytest.mark.gpu
def test_device_batch_above_one_chunk(orc):
    """more than 65 536 candidates: the call is cut into chunks of the internal 16-bit rate index"""
    rng = np.random.default_rng(500)
    fr, visits, jobs, states, ns = _kernel_case(rng, 10, 'noise')
    want = oracle(orc, fr, visits, jobs, states, ns)
    reps = -(-70000 // len(jobs))
    big = np.tile(jobs, reps)
    big['offset'] += np.repeat(np.arange(reps, dtype=np.uint32) * ns, len(jobs))
    with CE._engine(fr) as eng:
        got = eng.chroma_tu_eval(visits, big, ns * reps, states=states, want_level=True, want_reco=True)
    assert len(big) > 65536
    assert got['results'].tobytes() == np.tile(want['results'], reps).tobytes()
    assert np.array_equal(got['level'], np.tile(want['level'], reps)) and np.array_equal(got['reco'], np.tile(want['reco'], reps))


@pytest.mark.gpu
@pytest.mark.parametrize('bd', (8, 9, 10))
def test_device_extreme_qps_with_saturated_residuals(orc, bd):
    """chroma QP 0 and the maximum for the bit depth on pictures whose residuals reach +-(2^bd - 1)"""
    rng = np.random.default_rng(600 + bd)
    mx = (1 << bd) - 1
    fr = CE.Frame(rng, bd, 160, 128, 'noise')
    fr.cb[:], fr.cb_reco[:], fr.cr[:], fr.cr_reco[:], fr.luma[:] = mx, 0, 0, mx, 0    # Cb residuals +(2^bd - 1), Cr residuals -(2^bd - 1)
    visits = CE.make_visits(rng)
    states = random_states(rng, 8)
    jobs, ns = make_jobs(rng, visits, bd, per_visit=2, qps=(0, max_qp(bd)))
    want = oracle(orc, fr, visits, jobs, states, ns)
    compare(run_device(fr, visits, jobs, states, ns), want, '%d-bit extreme QP' % bd)
    full = 0
    for j in jobs:
        v = visits[j['visit']]
        n = 1 << (int(v['log2w']) + int(v['log2h']))
        full += int((want['pred'][j['offset']:j['offset'] + n] == 0).any()) + int((want['pred'][j['offset'] + n:j['offset'] + 2 * n] == mx).any())
    assert full > len(jobs)                                           # most candidates reach the full-scale residual in both components


@pytest.mark.gpu
def test_device_prediction_equals_chroma_eval(orc):
    rng = np.random.default_rng(700)
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = CE.make_visits(rng)
    jobs, ns = make_jobs(rng, visits, 10, per_visit=8, flags=(QUANT,))
    with CE._engine(fr) as eng:
        _, blocks = eng.chroma_eval(visits, want_pred=True)
        got = eng.chroma_tu_eval(visits, jobs, ns, want_pred=True)
    for j in jobs:
        b = blocks[j['visit']][j['cand']]
        assert np.array_equal(got['pred'][j['offset']:j['offset'] + b.size], b.ravel())


@pytest.mark.gpu
@pytest.mark.parametrize('dq', (0, 1))
def test_device_context_blind_equals_the_pinned_luma_tu_path(orc, dq):
    """uniform non-adapting models: each component's levels, reconstruction, SSE and bits equal vvcb_tu_eval's (DCT-II luma jobs on the
    same residual and prediction, the component's plane loaded as the luma picture)"""
    import vvc_intra_b200 as vb
    eng_mod = E()
    rng = np.random.default_rng(800 + dq)
    fr = CE.Frame(rng, 10, 160, 128, 'noise')
    visits = CE.make_visits(rng)
    flags = QUANT | RATE | (DEPQUANT if dq else 0)
    jobs, ns = make_jobs(rng, visits, 10, per_visit=2, flags=(flags,), n_states=1)
    cst = uniform_states(eng_mod.CHROMA_CTX_STATES_DTYPE, state=(20000, 9000))
    with CE._engine(fr) as eng:
        got = eng.chroma_tu_eval(visits, jobs, ns, states=cst, want_level=True, want_reco=True, want_pred=True)
    q = (20000 + 9000) >> 8
    rates = np.zeros(1, eng_mod.DQ_RATES_DTYPE)
    rv = rates.view(np.uint32).reshape(-1, 2)
    rv[:, 0], rv[:, 1] = FB[2 * q], FB[2 * q + 1]
    lst = uniform_states(eng_mod.CTX_STATES_DTYPE, state=(20000, 9000))
    delta = FB[2 * q + 1] - FB[2 * q]
    for c, (org, name) in enumerate(((fr.cb, 'Cb'), (fr.cr, 'Cr'))):
        tj = np.zeros(len(jobs), eng_mod.TU_JOB_DTYPE)
        resi = np.zeros(ns, np.int16)
        for i, j in enumerate(jobs):
            v = visits[j['visit']]
            w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
            o = j['offset'] + c * w * h
            p = got['pred'][o:o + w * h].reshape(h, w)
            resi[o:o + w * h] = (org[v['y']:v['y'] + h, v['x']:v['x'] + w].astype(np.int32) - p).ravel()
            t = tj[i]
            t['x'], t['y'], t['log2w'], t['log2h'], t['flags'] = v['x'], v['y'], v['log2w'], v['log2h'], flags
            t['qp_per'], t['qp_rem'], t['offset'], t['lambda'] = j['qp_per'][c], j['qp_rem'][c], o, j['lambda'][c]
            t['cbf_delta_bits'] = delta
        with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=CTU) as leng:
            leng.frame_begin(org)
            lo = leng.tu_eval(tj, resi, got['pred'], want_level=True, want_reco=True, rates=rates, states=lst)
        sel = np.zeros(ns, bool)
        for t in tj:
            sel[t['offset']:t['offset'] + (1 << (int(t['log2w']) + int(t['log2h'])))] = True
        assert np.array_equal(got['level'][sel], lo['level'][sel]), name
        assert np.array_equal(got['reco'][sel], lo['reco'][sel]), name
        comp = got['results']['comp'][:, c]
        for f in ('abs_sum_coeff', 'abs_sum_level', 'sse', 'frac_bits'):
            assert np.array_equal(comp[f], lo['results'][f]), (name, f)
        assert (comp['frac_bits'] > 0).sum() > len(jobs) // 2


@pytest.mark.gpu
def test_refusals(tmp_path):
    """every refusal returns its code and leaves the context usable; the broker proxy refuses the entry point"""
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
        rc = eng._lib.vvcb_chroma_tu_eval(eng._ctx, _p(visits), 2, _p(jobs), 1, _p(states), 2, ns, None, None, None,
                                          _p(np.zeros(1, eng_mod.CHROMA_TU_RESULT_DTYPE)))
        assert rc == -3                                               # before vvcb_chroma_frame_begin
        eng.reco_update(fr.luma)
        eng.chroma_frame_begin(fr.cb, fr.cr)
        ref = eng.chroma_tu_eval(visits, jobs, ns, states=states)['results']

        def call(v, j, st=states, n=ns):
            out = np.zeros(len(j), eng_mod.CHROMA_TU_RESULT_DTYPE)
            return eng._lib.vvcb_chroma_tu_eval(eng._ctx, _p(v), len(v), _p(j), len(j), _p(st) if st is not None else None,
                                                0 if st is None else len(st), n, None, None, None, _p(out))
        bad_jobs = []
        for f, val in (('visit', 2), ('cand', 8), ('flags', 0), ('flags', QUANT | 4), ('flags', QUANT | 8), ('flags', QUANT | 64),
                       ('rate_idx', 2), ('offset', ns - 1)):
            b = good.copy()
            b[f] = val
            bad_jobs.append(b)
        for c in range(2):
            for per, rem in ((-1, 0), (0, -1), (0, 6), (max_qp(10) // 6, max_qp(10) % 6 + 1), (13, 0)):
                b = good.copy()
                b['qp_per'][c], b['qp_rem'][c] = per, rem
                bad_jobs.append(b)
            for lam in (0.0, -1.0, float('inf'), float('nan')):
                b = good.copy()
                b['lambda'][c] = lam
                bad_jobs.append(b)
        lm_off = good.copy()
        lm_off['visit'], lm_off['cand'] = 1, 5                        # an LM candidate of a visit without cclm
        bad_jobs.append(lm_off)
        for b in bad_jobs:
            assert call(visits, np.array([good, b])) == -1, b
        assert call(visits, np.array([good]), st=None) == -1          # DEPQUANT / RATE without states
        bv = visits.copy()
        bv[1]['log2w'] = 6
        assert call(bv, np.array([good])) == -1                       # a visit vvcb_chroma_eval refuses
        dq_free = good.copy()
        dq_free['flags'], dq_free['lambda'] = QUANT, (0.0, 0.0)
        assert call(visits, np.array([dq_free]), st=None) == 0        # scalar quantisation needs neither lambda nor states
        assert eng.chroma_tu_eval(visits, jobs, ns, states=states)['results'].tobytes() == ref.tobytes()   # still usable
    # through the broker
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
                'j = np.zeros(1, E.CHROMA_TU_JOB_DTYPE); j["flags"] = 1\n'
                'try:\n'
                '    eng.chroma_tu_eval(np.zeros(1, E.CHROMA_VISIT_DTYPE), j, 64); print("accepted")\n'
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
