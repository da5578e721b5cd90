"""Evaluation of intra sub-partition (ISP) candidates whose blocks are at least 4x4 (vvcb_isp_eval).

The checker is the plain-C chain of tests/isp_oracle/isp_oracle.c on the oracle's pinned components.  The chaining itself (line
hand-over, cbf and context carry) is restated from the reference's code and NOT compared with the reference encoder's own ISP output;
what ties it down here: the literal shift-and-repeat hand-over equals the fresh fetch the kernel makes (CPU), the device equals the
chain bit for bit (GPU), and every block the chain codes equals the pinned TU path fed with the same prediction and models (GPU)."""
import ctypes as C
import os
import subprocess
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOR, VER = 1, 2


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as g
    g.build()
    L = C.CDLL(os.path.join(ROOT, 'tests/isp_oracle/libisp_oracle.so'))
    L.orc_isp_lines.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_int] * 11 + [C.c_void_p] * 3
    L.orc_ref_fill.argtypes = [C.c_void_p, C.c_int] + [C.c_int] * 11 + [C.c_void_p] * 2
    L.orc_isp_chain.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 9
    L.orc_isp_blocks.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return L


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def blocks(cu_w, cu_h, hor):
    """PartitionerImpl::getTUIntraSubPartitions: (number, block width, block height)"""
    split, other = (cu_h, cu_w) if hor else (cu_w, cu_h)
    size = max(split >> 2, 16 // other if other < 16 else 1)
    return split // size, (cu_w if hor else size), (size if hor else cu_h)


def in_scope():
    """every CU size x split whose blocks are all at least 4x4 (sizes up to 64, CU::canUseISP with a maximum TB size of 64)"""
    out = []
    for lw in range(2, 7):
        for lh in range(2, 7):
            if lw + lh <= 4:
                continue
            for isp in (HOR, VER):
                n, bw, bh = blocks(1 << lw, 1 << lh, isp == HOR)
                if bw >= 4 and bh >= 4:
                    out.append((1 << lw, 1 << lh, isp, n))
    return out


def test_scope_is_what_the_header_states():
    s = in_scope()
    assert all((h >= 16 or (w, h) == (4, 8)) for w, h, isp, _ in s if isp == HOR)
    assert all((w >= 16 or (w, h) == (8, 4)) for w, h, isp, _ in s if isp == VER)
    assert {n for *_, n in s} == {2, 4} and len(s) == 2 * (15 + 1)


def availabilities(w, h, rng):
    """all-or-nothing left / above, with the below-left and above-right prefixes they allow"""
    out = []
    for nl in (0, h // 4):
        for na in (0, w // 4):
            for al in (0, 1):
                nbl = int(rng.integers(0, h // 4 + 1)) if nl else 0
                nar = int(rng.integers(0, w // 4 + 1)) if na else 0
                out.append((al, na, nar, nl, nbl))
                if nl and na:
                    out.append((al, na, w // 4, nl, h // 4))
    return out


def _fresh_fetch(L, pic, stride, bd, x, y, w, h, hor, k, bw, bh, av, cu_reco):
    """block k as a fresh xFillReferenceSamples over a picture that holds blocks 0..k-1: lengths m_topRefLength / m_leftRefLength and
    availability derived from the CU's (include/vvc_intra_b200.h, vvcb_isp_eval)"""
    al, na, nar, nl, nbl = av
    T, Lh = w + bw, h + bh
    bx, by = (0, k * bh) if hor else (k * bw, 0)
    p = pic.copy()
    for j in range(k):
        jx, jy = (0, j * bh) if hor else (j * bw, 0)
        p[y + jy:y + jy + bh, x + jx:x + jx + bw] = cu_reco[j * bw * bh:(j + 1) * bw * bh].reshape(bh, bw)
    if k == 0:
        top_n, left_n, corner = 4 * (na + nar if na else 0), 4 * (nl + nbl if nl else 0), al
    elif hor:
        top_n, left_n, corner = w, (h + 4 * nbl - by) if nl else 0, int(nl > 0)
    else:
        top_n, left_n, corner = (w + 4 * nar - bx) if na else 0, h, int(na > 0)
    top_n, left_n = max(0, min(top_n, T)), max(0, min(left_n, Lh))
    wq, hq = T // 2, Lh // 2                            # orc_ref_fill fetches 2w / 2h samples: lengths T and L
    ua, ul = min(top_n // 4, wq >> 2), min(left_n // 4, hq >> 2)
    top = np.zeros(2 * wq + 1, np.int16)
    left = np.zeros(2 * hq + 1, np.int16)
    L.orc_ref_fill(_p(p), stride, x + bx, y + by, wq, hq, 0, bd, corner, ua, top_n // 4 - ua, ul, left_n // 4 - ul, _p(top), _p(left))
    return top, left


@pytest.mark.parametrize('bd', (8, 10))
def test_handover_formulations_agree(lib, bd):
    """The literal hand-over (orc_isp_lines: shift the held side, re-fetch the new line, repeat its last sample) equals a fresh fetch of
    block k with the derived lengths and availability -- the formulation isp_pred_kernel implements -- for every in-scope CU size x split
    x block x all-or-nothing availability, with random reconstructions."""
    rng = np.random.default_rng(bd)
    stride = 200
    checked = 0
    for w, h, isp, n in in_scope():
        _, bw, bh = blocks(w, h, isp == HOR)
        for av in availabilities(w, h, rng):
            pic = rng.integers(0, 1 << bd, (200, stride)).astype(np.int16)
            cu_reco = rng.integers(0, 1 << bd, w * h).astype(np.int16)
            x, y = 64, 64
            for k in range(n):
                T, Lh = w + bw, h + bh
                top = np.zeros(T + 1, np.int16)
                left = np.zeros(Lh + 1, np.int16)
                lib.orc_isp_lines(_p(pic), stride, bd, x, y, w, h, int(isp == HOR), k, *av, _p(cu_reco), _p(top), _p(left))
                ftop, fleft = _fresh_fetch(lib, pic, stride, bd, x, y, w, h, isp == HOR, k, bw, bh, av, cu_reco)
                assert top.tolist() == ftop[:T + 1].tolist(), (w, h, isp, k, av, 'top')
                assert left.tolist() == fleft[:Lh + 1].tolist(), (w, h, isp, k, av, 'left')
                checked += 1
    assert checked > 400


def test_block0_is_the_cu_fetch(lib):
    """block 0's lines are the CU-level orc_ref_fill over fetch_top_len / fetch_left_len (vvcb_isp_plan), cut to the block's lengths"""
    rng = np.random.default_rng(3)
    for w, h, isp, n in in_scope():
        _, bw, bh = blocks(w, h, isp == HOR)
        for av in availabilities(w, h, rng):
            pic = rng.integers(0, 1024, (200, 200)).astype(np.int16)
            top = np.zeros(w + bw + 1, np.int16)
            left = np.zeros(h + bh + 1, np.int16)
            lib.orc_isp_lines(_p(pic), 200, 10, 64, 64, w, h, int(isp == HOR), 0, *av, None, _p(top), _p(left))
            ctop, cleft = np.zeros(2 * w + 1, np.int16), np.zeros(2 * h + 1, np.int16)
            lib.orc_ref_fill(_p(pic), 200, 64, 64, w, h, 0, 10, *av, _p(ctop), _p(cleft))
            assert top.tolist() == ctop[:w + bw + 1].tolist() and left.tolist() == cleft[:h + bh + 1].tolist()


def test_struct_sizes_match_header(tmp_path):
    import vvc_intra_b200.engine as E
    src = tmp_path / 'sz.c'
    src.write_text('#include "vvc_intra_b200.h"\n#include <stdio.h>\n#include <stddef.h>\n'
                   'int main(void){printf("%zu %zu %zu %zu\\n", sizeof(vvcb_isp_job), sizeof(vvcb_isp_result),'
                   ' offsetof(vvcb_isp_job, cbf), offsetof(vvcb_isp_result, cbf_bits));return 0;}\n')
    exe = tmp_path / 'sz'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [E.ISP_JOB_DTYPE.itemsize, E.ISP_RESULT_DTYPE.itemsize, E.ISP_JOB_DTYPE.fields['cbf'][1],
                   E.ISP_RESULT_DTYPE.fields['cbf_bits'][1]]


# ---------------------------------------------------------------------------------------------------------------------------------
# device
# ---------------------------------------------------------------------------------------------------------------------------------
def random_states(rng, n):
    import vvc_intra_b200.engine as E
    s = np.zeros(n, E.CTX_STATES_DTYPE)
    flat = s.view(np.uint8).reshape(n, -1).view(np.uint16).reshape(n, -1, 3)     # per model: state0, state1, rate | pad << 8
    m = flat.shape[1]
    flat[:, :, 0] = rng.integers(1, 0x400, (n, m)) << 5
    flat[:, :, 1] = rng.integers(1, 0x4000, (n, m)) << 1
    flat[:, :, 2] = (rng.integers(4, 8, (n, m)) << 4) | rng.integers(4, 8, (n, m))
    return s


def random_models(rng):
    return [((int(rng.integers(1, 0x400)) << 5, int(rng.integers(1, 0x4000)) << 1), (int(rng.integers(4, 8)) << 4) | int(rng.integers(4, 8)), 0)
            for _ in range(2)]


class Frame:
    """a picture with the CUs laid out on a grid of 64x64 cells (each CU at its cell's origin + 64: neighbours inside the picture)"""

    def __init__(self, rng, bd, n_cells, extremes=True):
        import vvc_intra_b200.engine as E
        self.bd, self.cols = bd, 16
        rows = (n_cells + self.cols - 1) // self.cols
        self.h, self.w = 128 * rows + 64, 128 * self.cols + 64
        mx = (1 << bd) - 1
        self.orig = rng.integers(0, mx + 1, (self.h, self.w)).astype(np.int16)
        self.reco = np.clip(self.orig + rng.integers(-20, 21, self.orig.shape), 0, mx).astype(np.int16)
        self.visits = np.zeros(n_cells, E.VISIT_DTYPE)
        self.E = E
        if extremes:                                  # flat 0, flat max, +-max checkerboard in the first cells
            for c, kind in zip(range(min(3, n_cells)), ('zero', 'max', 'check')):
                y, x = self.cell(c)
                blk = np.zeros((192, 192), np.int16) if kind == 'zero' else np.full((192, 192), mx, np.int16)
                if kind == 'check':
                    blk = np.where((np.add.outer(np.arange(192), np.arange(192)) & 1) == 0, mx, 0).astype(np.int16)
                self.orig[y - 64:y + 128, x - 64:x + 128] = blk
                self.reco[y - 64:y + 128, x - 64:x + 128] = mx - blk if kind == 'check' else blk

    def cell(self, c):
        return 128 * (c // self.cols) + 64, 128 * (c % self.cols) + 64

    def set_cu(self, c, w, h, av):
        y, x = self.cell(c)
        v = self.visits[c]
        v['x'], v['y'], v['log2w'], v['log2h'] = x, y, w.bit_length() - 1, h.bit_length() - 1
        v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = av
        v['flags'] = 3


def _pick(v, i):
    return v[i] if isinstance(v, (list, tuple, np.ndarray)) else v


def make_batch(rng, bd, cases, dq, rate=True, use_mts=1):
    """cases: (w, h, isp, mode, qp, availability) -> frame, jobs, states, n_samples; dq / rate / use_mts: one value for the batch, or one
    per case"""
    E = __import__('vvc_intra_b200.engine', fromlist=['x'])
    fr = Frame(rng, bd, len(cases))
    jobs = np.zeros(len(cases), E.ISP_JOB_DTYPE)
    states = random_states(rng, len(cases))
    off = 0
    for i, (w, h, isp, mode, qp, av) in enumerate(cases):
        fr.set_cu(i, w, h, av)
        j = jobs[i]
        j['visit'], j['isp_mode'], j['mode'] = i, isp, mode
        j['flags'] = 1 | (2 if _pick(dq, i) else 0) | (32 if _pick(rate, i) else 0)
        j['use_mts'], j['max_tb_size'] = _pick(use_mts, i), 64
        j['qp_per'], j['qp_rem'], j['rate_idx'], j['offset'] = qp // 6, qp % 6, i, off
        for t, (st, r, pad) in enumerate(random_models(rng)):
            j['cbf'][t]['state'] = st
            j['cbf'][t]['rate'] = r
        j['lambda'] = 0.57 * 2.0 ** ((qp - 6 * (bd - 8) - 12) / 3.0)
        off += w * h
    return fr, jobs, states, off


def oracle_batch(lib, fr, jobs, states, n_samples, dep_quant=1):
    E = fr.E
    pred, level, reco = np.zeros(n_samples, np.int16), np.zeros(n_samples, np.int32), np.zeros(n_samples, np.int16)
    res = np.zeros(len(jobs), E.ISP_RESULT_DTYPE)
    carried = np.zeros((len(jobs), 4), E.CTX_STATES_DTYPE)
    delta = np.zeros((len(jobs), 4), np.int32)
    orig, reco_pic = np.ascontiguousarray(fr.orig), np.ascontiguousarray(fr.reco)
    for i, j in enumerate(jobs):
        v = fr.visits[j['visit']]
        o = int(j['offset'])
        n = (1 << int(v['log2w'])) * (1 << int(v['log2h']))
        pv, lv, rv = pred[o:o + n], level[o:o + n], reco[o:o + n]
        r, cs, d = res[i:i + 1], carried[i], delta[i]
        lib.orc_isp_chain(_p(orig), _p(reco_pic), fr.w, fr.bd, dep_quant, _p(fr.visits[j['visit']:j['visit'] + 1]), _p(jobs[i:i + 1]),
                          _p(states[j['rate_idx']:j['rate_idx'] + 1]), _p(pv), _p(lv), _p(rv), _p(r), _p(cs), _p(d))
    return dict(results=res, pred=pred, level=level, reco=reco, carried=carried, delta=delta)


def run_device(fr, jobs, states, n_samples):
    import vvc_intra_b200 as vb
    with vb.IntraCostEngine(device=0, bit_depth=fr.bd, ctu_size=128) as eng:
        eng.frame_begin(fr.orig)
        eng.reco_update(fr.reco)
        return eng.isp_eval(fr.visits, jobs, n_samples, states=states, want_level=True, want_reco=True, want_pred=True)


def compare(dev, ora, what=''):
    for key in ('pred', 'level', 'reco'):
        bad = np.flatnonzero(dev[key] != ora[key])
        assert bad.size == 0, (what, key, bad[:5])
    d, o = dev['results'], ora['results']
    for f in ('n_parts', 'cbf', 'cbf_bits', 'discarded'):
        assert np.array_equal(d[f], o[f]), (what, f, np.flatnonzero((d[f] != o[f]).reshape(len(d), -1).any(1))[:5])
    for f in ('abs_sum_coeff', 'abs_sum_level', 'sse', 'frac_bits'):
        assert np.array_equal(d['part'][f], o['part'][f]), (what, f, np.flatnonzero((d['part'][f] != o['part'][f]).any(1))[:5])


def all_mode_cases(rng, bd):
    cases = []
    qps = (22, 27, 32, 37)
    for w, h, isp, n in in_scope():
        avs = availabilities(w, h, rng)
        for mode in range(67):
            av = avs[int(rng.integers(0, len(avs)))]
            cases.append((w, h, isp, mode, qps[len(cases) % 4] + 6 * (bd - 8), av))
    return cases


@pytest.mark.gpu
@pytest.mark.parametrize('bd,dq', [(8, 0), (8, 1), (10, 0), (10, 1)])
def test_device_matches_oracle_chain(lib, bd, dq):
    """every in-scope CU shape x split x all 67 modes, QPs 22 / 27 / 32 / 37, random all-or-nothing availability, extreme pictures in the
    first cells; two- and four-block candidates mixed in one batch"""
    rng = np.random.default_rng(100 * bd + dq)
    cases = all_mode_cases(rng, bd)
    fr, jobs, states, ns = make_batch(rng, bd, cases, dq)
    dev = run_device(fr, jobs, states, ns)
    ora = oracle_batch(lib, fr, jobs, states, ns)
    assert set(ora['results']['n_parts'].tolist()) == {2, 4}
    compare(dev, ora, (bd, dq))


@pytest.mark.gpu
def test_mixed_batch_matches_oracle_chain(lib):
    """one batch mixing scalar and dependent quantisation, candidates with and without VVCB_TU_RATE and with and without MTS (DCT-II in
    both directions), every in-scope shape x split: pass 1 skips the scalar candidates and only some candidates carry models"""
    rng = np.random.default_rng(21)
    bd = 10
    cases = [c for c in all_mode_cases(rng, bd) if rng.random() < 0.3]
    n = len(cases)
    dq, rate, mts = (rng.integers(0, 2, n).tolist() for _ in range(3))
    fr, jobs, states, ns = make_batch(rng, bd, cases, dq, rate=rate, use_mts=mts)
    assert len({(a, b, c) for a, b, c in zip(dq, rate, mts)}) == 8
    dev = run_device(fr, jobs, states, ns)
    ora = oracle_batch(lib, fr, jobs, states, ns)
    compare(dev, ora, 'mixed')
    assert not dev['results']['part']['frac_bits'][np.array(rate) == 0].any()


@pytest.mark.gpu
@pytest.mark.parametrize('dq', (0, 1))
def test_blocks_match_the_pinned_tu_path(lib, dq):
    """Each block of a sample of candidates, fed to vvcb_tu_eval with the prediction vvcb_isp_eval returned, the models the previous
    block left (oracle chain), their prices and the chain's cbfDeltaBits, where the transform pair has a public mts_idx (DCT-II x DCT-II: 0,
    DST-VII x DST-VII: 2): levels, SSE and residual bits equal bit for bit."""
    import vvc_intra_b200 as vb
    E = vb.engine
    rng = np.random.default_rng(7 + dq)
    bd = 10
    cases = [c for c in all_mode_cases(rng, bd) if rng.random() < 0.25]
    fr, jobs, states, ns = make_batch(rng, bd, cases, dq)
    dev = run_device(fr, jobs, states, ns)
    ora = oracle_batch(lib, fr, jobs, states, ns)
    tj, st, resi, pred, want = [], [], [], [], []
    off = 0
    for i, (w, h, isp, mode, qp, av) in enumerate(cases):
        n, bw, bh = blocks(w, h, isp == HOR)
        dst = (bw <= 16, bh <= 16)
        if dst[0] != dst[1]:
            continue
        v = fr.visits[i]
        for k in range(n):
            bx, by = (0, k * bh) if isp == HOR else (k * bw, 0)
            o = int(jobs[i]['offset']) + k * bw * bh
            p = dev['pred'][o:o + bw * bh]
            org = fr.orig[v['y'] + by:v['y'] + by + bh, v['x'] + bx:v['x'] + bx + bw].ravel()
            j = np.zeros(1, E.TU_JOB_DTYPE)[0]
            j['x'], j['y'], j['log2w'], j['log2h'] = v['x'] + bx, v['y'] + by, bw.bit_length() - 1, bh.bit_length() - 1
            j['mts_idx'] = 2 if dst[0] else 0
            j['flags'] = 1 | 32 | (2 if dq else 0)
            j['qp_per'], j['qp_rem'], j['offset'], j['rate_idx'] = qp // 6, qp % 6, off, len(tj)
            j['cbf_delta_bits'], j['lambda'] = ora['delta'][i][k], jobs[i]['lambda']
            tj.append(j)
            st.append(states[i] if k == 0 else ora['carried'][i][k - 1])
            resi.append((org.astype(np.int32) - p).astype(np.int16))
            pred.append(p)
            want.append((i, k, o, bw * bh))
            off += bw * bh
    st = np.array(st, E.CTX_STATES_DTYPE)
    rates = np.zeros(len(st), E.DQ_RATES_DTYPE)
    for r, s in zip(rates.view(np.uint32).reshape(len(st), -1), st.view(np.uint8).reshape(len(st), -1).view(np.uint16).reshape(len(st), -1, 3)[:, 11:]):
        q = (s[:, 0].astype(np.int64) + s[:, 1]) >> 8
        fb = np.array(fracbits_table(lib), np.uint32)
        r[0::2], r[1::2] = fb[2 * q], fb[2 * q + 1]
    with vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=128) as eng:
        eng.frame_begin(fr.orig)
        out = eng.tu_eval(np.array(tj, E.TU_JOB_DTYPE), np.concatenate(resi), np.concatenate(pred), want_level=True, rates=rates, states=st)
    assert len(want) > 100
    for t, (i, k, o, n) in enumerate(want):
        lo = int(tj[t]['offset'])
        assert out['level'][lo:lo + n].tolist() == dev['level'][o:o + n].tolist(), (i, k)
        r = out['results'][t]
        p = dev['results'][i]['part'][k]
        assert (r['sse'], r['frac_bits'], r['abs_sum_level']) == (p['sse'], p['frac_bits'], p['abs_sum_level']), (i, k)


_FB = None


def fracbits_table(lib):
    """ProbModelTables::m_binFracBits, read back through the oracle's rate: intBits of a context from its state (orc_rates_from_states)"""
    global _FB
    if _FB is None:
        import vvc_intra_b200.engine as E
        lib.orc_rates_from_states.argtypes = [C.c_void_p, C.c_void_p]
        tab = [0] * 512
        for q in range(256):
            s = np.zeros(1, E.CTX_STATES_DTYPE)
            s.view(np.uint8).view(np.uint16)[3 * 11:3 * 11 + 2] = (q << 7, q << 7)       # first priced model: state sum >> 8 == q
            r = np.zeros(1, E.DQ_RATES_DTYPE)
            lib.orc_rates_from_states(_p(s), _p(r))
            tab[2 * q], tab[2 * q + 1] = (int(v) for v in r.view(np.uint32)[:2])
        _FB = tab
    return _FB


@pytest.mark.gpu
def test_walk_and_sweep_batches_agree():
    """the same candidates alone, in a walk-sized batch (~40) and inside a sweep-sized batch (>= 100 000: the dependent quantiser's sorted
    path) give identical results"""
    rng = np.random.default_rng(11)
    bd = 10
    base = [(w, h, isp, int(rng.integers(0, 67)), 32, (1, w // 4, 0, h // 4, 0)) for w, h, isp, n in in_scope() if w * h <= 256]
    walk = (base * 3)[:40]
    fr, jobs, states, ns = make_batch(rng, bd, walk, dq=1)
    ref = run_device(fr, jobs, states, ns)
    one = run_device(fr, jobs[:1], states, int(jobs[1]['offset']))
    assert one['results'].tobytes() == ref['results'][:1].tobytes()
    reps = (100000 + len(walk) - 1) // len(walk)
    big = np.concatenate([jobs] * reps)
    big['offset'] = np.arange(len(big)) // len(walk) * ns + np.tile(jobs['offset'], reps)
    out = run_device(fr, big, states, ns * reps)
    assert len(big) >= 100000
    for r in range(0, reps, max(1, reps // 7)):
        assert out['results'][r * len(walk):(r + 1) * len(walk)].tobytes() == ref['results'].tobytes(), r
        assert np.array_equal(out['level'][r * ns:(r + 1) * ns], ref['level'])


@pytest.mark.gpu
def test_refusals():
    """every VVCB_ERR_ARG case of vvcb_isp_eval.  GPU only by necessity: an engine context needs a CUDA device (vvcb_create fails without
    one), so no CPU run can reach the argument checks."""
    import vvc_intra_b200 as vb
    rng = np.random.default_rng(5)
    fr, jobs, states, ns = make_batch(rng, 10, [(16, 16, HOR, 18, 32, (1, 4, 0, 4, 0)), (16, 8, VER, 2, 32, (1, 4, 0, 2, 0))], dq=1)
    bad_visits = fr.visits.copy()

    def edit(fn, visits=None, n_samples=ns, st=states):
        j = jobs.copy()
        fn(j)
        return j, (fr.visits if visits is None else visits), n_samples, st

    def set_(f, v):
        return lambda j: j[0].__setitem__(f, v)

    cases = [edit(set_('isp_mode', 0)), edit(set_('isp_mode', 3)),
             edit(set_('mode', 67)),
             edit(set_('lfnst_idx', 1)), edit(set_('flags', 1 | 4)), edit(set_('flags', 1 | 8)), edit(set_('flags', 1 | 16)), edit(set_('flags', 2)),
             edit(set_('rate_idx', 2)), edit(set_('lambda', 0.0)), edit(set_('visit', 5)), edit(set_('max_tb_size', 8)),
             edit(lambda j: None, n_samples=ns - 1), edit(lambda j: None, st=None)]
    bv = bad_visits.copy(); bv[0]['n_left'] = 2
    cases.append(edit(lambda j: None, visits=bv))
    bv = bad_visits.copy(); bv[0]['n_above'] = 0; bv[0]['n_above_right'] = 1
    cases.append(edit(lambda j: None, visits=bv))
    bv = bad_visits.copy(); bv[1]['log2w'] = 3; bv[1]['log2h'] = 3          # 8x8: blocks of two samples either way
    cases.append(edit(lambda j: None, visits=bv))
    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=128) as eng:
        eng.frame_begin(fr.orig)
        eng.reco_update(fr.reco)
        eng.isp_eval(fr.visits, jobs, ns, states=states)                   # the unedited batch is accepted
        for j, visits, n_samples, st in cases:
            with pytest.raises(vb.engine.EngineError):
                eng.isp_eval(visits, j, n_samples, states=st)


# ---------------------------------------------------------------------------------------------------------------------------------
# the kernel source on host threads (tests/host_emul/cuda_emul.h)
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp('emul_isp') / 'libemul_isp.so'
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-g', '-ffp-contract=off', '-fPIC', '-shared', '-pthread', '-Wall', '-Wno-unused-function',
                           '-Wno-unknown-pragmas', '-Wno-unused-variable', '-o', str(out), os.path.join(ROOT, 'tests/host_emul/emul_isp.cpp')])
    L = C.CDLL(str(out))
    L.emul_isp_pred.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    return L


def wide_modes(w, h):
    """the modes PU::getWideAngIntraMode remaps for the CU's shape"""
    d = abs(w.bit_length() - h.bit_length())
    shift = (0, 6, 10, 12, 14, 15)[d]
    return list(range(2, 2 + shift)) if w > h else (list(range(67 - shift, 67)) if h > w else [])


def test_emulated_isp_pred_kernel_matches_oracle_chain(lib, emul):
    """isp_pred_kernel (the kernel source, compiled for host threads) predicts every block of seeded candidates of every in-scope shape x
    split -- modes 0, 1, 2, 18, 34, 50, 66 and the shape's wide angles, random all-or-nothing availability -- from the reconstruction of
    the previous blocks that the oracle chain produced, and equals the chain's prediction and residual"""
    rng = np.random.default_rng(31)
    bd = 10
    cases = []
    for w, h, isp, n in in_scope():
        avs = availabilities(w, h, rng)
        for mode in sorted(set((0, 1, 2, 18, 34, 50, 66) + tuple(wide_modes(w, h)))):
            cases.append((w, h, isp, mode, 27 + 6 * (bd - 8), avs[int(rng.integers(0, len(avs)))]))
    fr, jobs, states, ns = make_batch(rng, bd, cases, dq=0, rate=False)
    ora = oracle_batch(lib, fr, jobs, states, ns)
    cand = np.zeros((len(cases), 12), np.int32)
    for i, (w, h, isp, mode, qp, av) in enumerate(cases):
        v = fr.visits[i]
        cand[i] = (v['x'], v['y'], w, h, int(isp == HOR), mode, *av, jobs[i]['offset'])
    orig, reco = np.ascontiguousarray(fr.orig), np.ascontiguousarray(fr.reco)
    pred, resi = np.zeros(ns, np.int16), np.zeros(ns, np.int16)
    for k in range(4):
        emul.emul_isp_pred(_p(orig), _p(reco), fr.w, bd, _p(cand), len(cases), k, _p(ora['reco']), _p(pred), _p(resi))
    bad = np.flatnonzero(pred != ora['pred'])
    assert bad.size == 0, [cases[int(np.searchsorted(jobs['offset'], b, side='right')) - 1][:4] for b in bad[:5]]
    for i, (w, h, isp, mode, qp, av) in enumerate(cases):
        n, bw, bh = blocks(w, h, isp == HOR)
        o, v = int(jobs[i]['offset']), fr.visits[i]
        for k in range(n):
            bx, by = (0, k * bh) if isp == HOR else (k * bw, 0)
            org = fr.orig[v['y'] + by:v['y'] + by + bh, v['x'] + bx:v['x'] + bx + bw].ravel().astype(np.int32)
            blk = slice(o + k * bw * bh, o + (k + 1) * bw * bh)
            assert np.array_equal(resi[blk], (org - ora['pred'][blk]).astype(np.int16)), (w, h, isp, mode, k)
    assert len(cases) > 400
