"""The TU stage at the ends of its ranges: every internal QP from 0 to 63 + 6 (bitDepth - 8) at 8, 9 and 10 bit, full-scale residuals
(flat, checkerboard and stripes at +-max, impulses, full-range noise) and hand-built level blocks at +-32767 / -32768, against the oracle
byte for byte.  Each case set also asserts that it reached the edge it is there for (16-bit levels, the dependent quantiser's maxQIdx
clamp and dequantiser clip, the limited prefix of the Rice / exp-Golomb escape, 64-bit SSE above 2^31, the dependent quantiser's
shift count of 64 and more), from small replicas of the kernels' conditions, so that the cases cannot silently stop reaching it.

GPU tier: vvcb_tu_eval and vvcb_residual_bits.  CPU tier: a subset of the same cases through the kernel source on host threads
(tests/host_emul); the device-only branches of dq_init_quant (__dmul_rn, the device shift) run only in the GPU tier."""
import itertools

import numpy as np
import pytest

import vvc_intra_b200 as vb
from oracle import oracle_py as O
import golden_util as G
from test_kernel_emulation import run_emul_rate, run_emul_tu

BDS = (8, 9, 10)
SHAPES = [(lw, lh) for lw in range(2, 7) for lh in range(2, 7)]
FAMILIES = ('flat', 'check', 'hstripe', 'vstripe', 'impulse_last', 'noise', 'isolated', 'zero_resi')
LAMBDA_SCALES = (0.25, 1.0, 4.0)
LFNST_MODES = (0, 1, 8, 18, 34, 50, 60, 66)          # LFNST sets 0 (planar, DC), 1 (2..12, 56..66), 2 (13..23, 45..55), 3 (24..44)
N_RATES = 5
QUANT_SCALES = (26214, 23302, 20560, 18396, 16384, 14564, 18396, 16384, 14564, 13107, 11651, 10280)   # g_quantScales
GO_RICE_PARS = np.array([0] * 7 + [1] * 7 + [2] * 14 + [3] * 4)                                       # g_goRiceParsCoeff
TS_RICE_PARS = np.array([0] * 12 + [1] * 13 + [2] * 7)                                                  # tsRicePars of vvcb_romfill.h


def max_qp(bd):
    return 63 + 6 * (bd - 8)


def qp_list(bd):
    """0, 1, 5, 6, 11, 12, both sides of every qp_per boundary, 51 + QpBdOffset and the top value"""
    top = max_qp(bd)
    s = {0, 1, 5, 6, 11, 12, 51 + 6 * (bd - 8), top}
    for k in range(1, top // 6 + 1):
        s |= {6 * k - 1, 6 * k}
    return sorted(q for q in s if q <= top)


def ref_lambda(qp, scale):
    """0.57 * 2^((QP - 12) / 3) on the internal QP (QpBdOffset included): the recorded lambdas of the *_depquant fixtures are this
    value times the reference's intra factor 1.0595 at 8 and at 10 bit"""
    return scale * 0.57 * 2.0 ** ((qp - 12) / 3.0)


# ---- content ----------------------------------------------------------------------------------------------------------------------
def content(fam, w, h, bd, sign, rng):
    """-> (pred, org, resi) int16.  resi is what the kernel transforms; org is what SSE is measured against."""
    mx = (1 << bd) - 1
    y, x = np.mgrid[0:h, 0:w]
    if fam == 'noise':
        pred = rng.integers(0, mx + 1, (h, w))
        org = rng.integers(0, mx + 1, (h, w))
        resi = org - pred
    elif fam == 'zero_resi':                       # nothing to code, org != pred: SSE = w * h * mx^2 (> 2^31 on a 64x64 10-bit block)
        pred = np.full((h, w), 0 if sign > 0 else mx)
        org = mx - pred
        resi = np.zeros((h, w), np.int64)
    else:
        if fam == 'flat':                          # saturates DC
            pat = np.ones((h, w), np.int64)
        elif fam == 'check':                       # the largest high-frequency coefficients and first-stage intermediates
            pat = 1 - 2 * ((x + y) & 1)
        elif fam == 'hstripe':
            pat = 1 - 2 * (y & 1)
        elif fam == 'vstripe':
            pat = 1 - 2 * (x & 1)
        elif fam == 'impulse_last':                # the last position of the up-right diagonal scan
            pat = ((x == w - 1) & (y == h - 1)).astype(np.int64)
        else:                                      # 'isolated': one sample, zero template around it
            pat = ((x == int(rng.integers(0, w))) & (y == int(rng.integers(0, h)))).astype(np.int64)
        resi = sign * mx * pat
        pred = np.where(resi > 0, 0, np.where(resi < 0, mx, mx // 2))
        org = pred + resi
    return pred.astype(np.int16), org.astype(np.int16), resi.astype(np.int16)


def chain_specs(chain, corners):
    """(log2w, log2h, mts_idx, lfnst_idx) each quantiser accepts; corners: the shapes crossed with every QP and family"""
    if corners:
        return {'scalar': [(2, 2, 0, 0), (6, 6, 0, 0), (5, 5, 1, 0)], 'dq': [(2, 2, 0, 0), (6, 6, 0, 0), (3, 3, 0, 2)],
                'rdoq': [(2, 2, 1, 0), (5, 5, 1, 0)]}[chain]
    out = []
    for lw, lh in SHAPES:
        small = lw <= 5 and lh <= 5
        if chain == 'scalar':
            out += [(lw, lh, m, 0) for m in (range(6) if small else (0,))]
        elif chain == 'dq':
            out += [(lw, lh, m, 0) for m in ((0, 2, 3, 4, 5) if small else (0,))] + [(lw, lh, 0, 1), (lw, lh, 0, 2)]
        elif small:
            out.append((lw, lh, 1, 0))
    return out


def tu_cases(rng, bd, chain, corner_qps=None, sweep=True):
    """Items for G.oracle_tu_chain / oracle_dq_chain / oracle_rdoq_chain and their jobs: every (shape, transform, LFNST) of the chain x
    every family with the QP list cycled through, plus the corner shapes x every family x every QP of corner_qps (default: all).  Every
    job carries VVCB_TU_RATE.  Returns (orig, jobs, resi, pred, rates, states, items)."""
    qps = qp_list(bd)
    corner_qps = qps if corner_qps is None else corner_qps
    todo = [(s, f, qps[(k * 5) % len(qps)]) for k, (s, f) in enumerate(itertools.product(chain_specs(chain, False), FAMILIES))] if sweep else []
    todo += [(s, f, q) for s, f, q in itertools.product(chain_specs(chain, True), FAMILIES, corner_qps)]
    rates = np.zeros(N_RATES, vb.DQ_RATES_DTYPE)
    for name in rates.dtype.names:
        rates[name] = rng.integers(300, 140000, rates[name].shape)
    states = np.zeros(N_RATES, vb.CTX_STATES_DTYPE)
    flat = states.view(vb.BIN_MODEL_DTYPE).reshape(N_RATES, -1)
    flat['state'][..., 0] = rng.integers(1, 1023, flat.shape) << 5                  # MASK_0 domain
    flat['state'][..., 1] = rng.integers(1, 16383, flat.shape) << 1                 # MASK_1 domain
    flat['rate'] = (rng.integers(4, 8, flat.shape) << 4) | rng.integers(4, 10, flat.shape)
    quant = {'scalar': vb.TU_QUANT, 'dq': vb.TU_QUANT | vb.TU_DEPQUANT, 'rdoq': vb.TU_QUANT | vb.TU_RDOQ_TS}[chain]
    items = []
    for k, ((lw, lh, mts, lfnst), fam, qp) in enumerate(todo):
        w, h = 1 << lw, 1 << lh
        pred, org, resi = content(fam, w, h, bd, 1 if k % 2 else -1, rng)
        small = lw <= 5 and lh <= 5
        flags = quant | vb.TU_RATE | (vb.TU_TS_ALLOWED | vb.TU_MTS_ALLOWED if small else 0)
        ri = k % N_RATES
        it = dict(pred=pred, org=org, resi=resi, mts=mts, lfnst=lfnst, intra=LFNST_MODES[k % len(LFNST_MODES)] if lfnst else 0, qp=qp,
                  per=qp // 6, rem=qp % 6, lam=ref_lambda(qp, LAMBDA_SCALES[k % 3]), cbf=int(rng.integers(-40000, 40000)), rate_idx=ri,
                  rate=rates[ri], flags=flags, fam=fam)
        it['bits_fn'] = (lambda lv, m=mts, s=small, st=states[ri]: O.residual_bits(lv, m, s, s, 1, st))
        items.append(it)
    n, cols = len(items), 16
    orig = np.zeros((64 * ((n + cols - 1) // cols + 1), 64 * cols), np.int16)
    jobs = np.zeros(n, vb.TU_JOB_DTYPE)
    off = 0
    for i, it in enumerate(items):
        h, w = it['resi'].shape
        cx, cy = 64 * (i % cols), 64 * (i // cols)
        orig[cy:cy + h, cx:cx + w] = it['org']
        j = jobs[i]
        j['x'], j['y'], j['log2w'], j['log2h'], j['mts_idx'], j['flags'] = cx, cy, w.bit_length() - 1, h.bit_length() - 1, it['mts'], it['flags']
        j['qp_per'], j['qp_rem'], j['offset'], j['rate_idx'] = it['per'], it['rem'], off, it['rate_idx']
        j['lfnst_idx'], j['intra_mode'], j['cbf_delta_bits'], j['lambda'] = it['lfnst'], it['intra'], it['cbf'], it['lam']
        it['off'] = off
        off += w * h
    return (orig, jobs, np.concatenate([it['resi'].ravel() for it in items]), np.concatenate([it['pred'].ravel() for it in items]),
            rates, states, items)


ORACLE_CHAIN = {'scalar': G.oracle_tu_chain, 'dq': G.oracle_dq_chain, 'rdoq': G.oracle_rdoq_chain}


def assert_same(out, exp, items):
    for k in ('coeff', 'level', 'reco'):
        bad = [i for i, it in enumerate(items) if not np.array_equal(out[k][it['off']:it['off'] + it['resi'].size], exp[k][it['off']:it['off'] + it['resi'].size])]
        assert not bad, (k, len(bad), [(items[i]['resi'].shape, items[i]['mts'], items[i]['lfnst'], items[i]['qp'], items[i]['fam']) for i in bad[:5]])
    n = len(items)
    bad = np.flatnonzero((out['results'].view(np.uint8).reshape(n, -1) != exp['results'].view(np.uint8).reshape(n, -1)).any(1))
    assert bad.size == 0, (len(bad), [(items[i]['resi'].shape, items[i]['mts'], items[i]['qp'], items[i]['fam'], out['results'][i], exp['results'][i]) for i in bad[:3]])


# ---- replicas of the kernels' conditions (reach) ------------------------------------------------------------------------------------
def limited_prefix(level, mts):
    """True when residual coding of this block certainly takes rate_rem_abs's limited-prefix branch ((bins >> rice) - 5 >= 2^12 - 1,
    vvcb_rate.cuh).  Transform skip: exact (mod >= 10 codes (mod - 10) >> 1 with the left / above Rice parameter).  Regular: a
    sufficient condition -- a remainder is at least (|level| - 4) >> 1 and its Rice parameter at most g_goRiceParsCoeff of the template sum."""
    a = np.abs(np.asarray(level, np.int64))
    h, w = a.shape
    if mts == 1:
        left, above = np.zeros_like(a), np.zeros_like(a)
        left[:, 1:], above[1:, :] = a[:, :-1], a[:-1, :]
        p1 = np.maximum(left, above)
        mod = np.where(a == p1, 1, np.where(a < p1, a + 1, a))
        return bool(((mod >= 10) & ((((mod - 10) >> 1) >> TS_RICE_PARS[np.minimum(left + above, 31)]) >= 4100)).any())
    p = np.zeros((h + 2, w + 2), np.int64)
    p[:h, :w] = a
    tmpl = p[:h, 1:w + 1] + p[:h, 2:w + 2] + p[1:h + 1, :w] + p[2:h + 2, :w] + p[1:h + 1, 1:w + 1]
    return bool(((a >= 4) & ((((a - 4) >> 1) >> GO_RICE_PARS[np.minimum(tmpl, 31)]) >= 4100)).any())


def dq_init_quant(bd, lw, lh, qp, lam):
    """Quantizer::initQuantBlock as dq_init_quant computes it (vvcb_dq.cuh): IEEE doubles, one rounding per operation"""
    qp_per = (qp + 1) // 6
    qp_rem = qp + 1 - 6 * qp_per
    nom = 15 - bd - ((lw + lh) >> 1)
    sqrt2 = (lw + lh) & 1
    tr = nom - sqrt2
    q_shift = 13 + qp_per + tr
    q_scale = QUANT_SCALES[sqrt2 * 6 + qp_rem]
    max_q_idx = (1 << (min(16, 32 + (7 - qp_per - tr) - 7) - 1)) - 4
    nom_d = 15 - 2 * nom + q_shift + sqrt2
    qs2 = float(q_scale * q_scale)
    den = qs2 * lam
    f = 1.0 / (float(1 << -nom_d) * den) if nom_d < 0 else float(1 << nom_d) / den
    pow2 = int(f * qs2) + 1
    dist_shift = 62 + q_shift - 30 - (pow2 - 1).bit_length()
    return dict(q_shift=q_shift, q_add=-((3 << q_shift) >> 1), q_scale=q_scale, max_q_idx=max_q_idx, count=dist_shift + q_shift, f=f)


def reach(items, exp, bd, chain):
    r = dict(lvl16=0, limited=0, sse31=0, clamp=0, deq_clip=0, shift64=0, ts_max=0, qps=set())
    for i, it in enumerate(items):
        h, w = it['resi'].shape
        sl = slice(it['off'], it['off'] + w * h)
        lv = exp['level'][sl].reshape(h, w)
        r['qps'].add(it['qp'])
        r['lvl16'] += int((np.abs(lv) == 32767).any())
        if it['mts'] == 1:
            r['ts_max'] = max(r['ts_max'], int(np.abs(lv).max()))
        r['limited'] += limited_prefix(lv, it['mts'])
        r['sse31'] += int(exp['results'][i]['sse']) > 2 ** 31
        if chain == 'dq':
            q = dq_init_quant(bd, w.bit_length() - 1, h.bit_length() - 1, it['qp'], it['lam'])
            q0 = (np.abs(exp['coeff'][sl].astype(np.int64)) * q['q_scale'] + q['q_add']) >> q['q_shift']
            r['clamp'] += int((q0 > q['max_q_idx']).any())
            deq = O.dep_dequant(lv, bd, it['qp'])
            r['deq_clip'] += int(((deq == 32767) | (deq == -32768)).any())
            if q['count'] >= 64:
                r['shift64'] += 1
                # the oracle (x86: count & 63) and the device (shift of 64 or more gives 0) round distStepAdd to the same 0
                assert int(q['f'] * float(1 << (q['count'] & 63)) + .5) == 0, (w, h, it['qp'], it['lam'], q['count'])
    return r


def assert_reach(r, bd, chain, all_qps=True):
    if all_qps:
        assert r['qps'] == set(qp_list(bd))
    if chain == 'rdoq':
        # transform-skip levels stay far below the limited prefix (its test is test_residual_bits_on_extreme_levels): the set reaches
        # the largest one instead, that of a +-max residual at QP 0
        mx = np.full((4, 4), (1 << bd) - 1, np.int16)
        assert r['ts_max'] >= int(O.quant_scalar(O.fwd_transform(mx, bd, 1), bd, 0, 0, True)[0].max()), r
    else:
        assert r['limited'] > 0, r
    if chain == 'scalar' and bd >= 9:
        assert r['lvl16'] > 0, r                   # trShift < 1 on 32x64 / 64x64 blocks: Quant::quant clips to +-32767
    if chain != 'rdoq' and bd == 10:
        assert r['sse31'] > 0, r
    if chain == 'dq':
        assert r['clamp'] > 0 and r['deq_clip'] > 0 and r['shift64'] > 0, r


# ---- stand-alone residual coding on hand-built level blocks -------------------------------------------------------------------------
LEVEL_FAMILIES = ('max', 'min', 'full', 'isolated', 'last')
ISOLATED = (8203, 8204, 8209, 8210, 32767, -32768)     # either side of the limited prefix, regular (8204) and transform skip (8210)


def level_cases(rng, shapes=SHAPES):
    jobs, levels, recs = [], [], []
    states = np.zeros(N_RATES, vb.CTX_STATES_DTYPE)
    flat = states.view(vb.BIN_MODEL_DTYPE).reshape(N_RATES, -1)
    flat['state'][..., 0] = rng.integers(1, 1023, flat.shape) << 5
    flat['state'][..., 1] = rng.integers(1, 16383, flat.shape) << 1
    flat['rate'] = (rng.integers(4, 8, flat.shape) << 4) | rng.integers(4, 10, flat.shape)
    off = 0
    for lw, lh in shapes:
        small = lw <= 5 and lh <= 5
        w, h = 1 << lw, 1 << lh
        for mts in (range(6) if small else (0,)):
            for fam in LEVEL_FAMILIES:
                for v in (ISOLATED if fam == 'isolated' else (None,)):
                    s = rng.choice([-1, 1], (h, w))
                    if fam == 'max':                   # every coefficient non-zero: the context-coded bin budget runs out
                        lv = 32767 * s
                    elif fam == 'min':
                        lv = np.full((h, w), -32768)
                    elif fam == 'full':
                        lv = rng.integers(1, 32768, (h, w)) * s
                        lv[rng.random((h, w)) < 0.1] = -32768
                    else:
                        lv = np.zeros((h, w), np.int64)
                        if fam == 'isolated':
                            lv[rng.integers(0, h), rng.integers(0, w)] = v
                        else:
                            lv[h - 1, w - 1] = 32767 * s[0, 0]
                    if max(w, h) == 64:                # only the low 32x32 of a 64-point side is coded
                        lv[32:, :] = 0
                        lv[:, 32:] = 0
                        if fam in ('isolated', 'last') and not lv.any():
                            lv[min(h, 32) - 1, min(w, 32) - 1] = v if v is not None else -32768
                    j = np.zeros(1, vb.TU_JOB_DTYPE)[0]
                    j['log2w'], j['log2h'], j['mts_idx'], j['offset'], j['rate_idx'] = lw, lh, mts, off, len(jobs) % N_RATES
                    j['flags'] = vb.TU_QUANT | vb.TU_RATE | (vb.TU_TS_ALLOWED | vb.TU_MTS_ALLOWED if small else 0)
                    jobs.append(j)
                    levels.append(lv.astype(np.int32))
                    recs.append((lw, lh, mts, fam, v))
                    off += w * h
    jobs = np.array(jobs, vb.TU_JOB_DTYPE)
    exp = [O.residual_bits(lv, int(j['mts_idx']), bool(j['flags'] & vb.TU_TS_ALLOWED), bool(j['flags'] & vb.TU_MTS_ALLOWED), 1,
                           states[int(j['rate_idx'])]) for lv, j in zip(levels, jobs)]
    return jobs, levels, states, recs, exp


def assert_level_reach(levels, jobs, recs):
    reg = sum(limited_prefix(lv, int(j['mts_idx'])) for lv, j in zip(levels, jobs) if j['mts_idx'] != 1)
    ts = sum(limited_prefix(lv, 1) for lv, j in zip(levels, jobs) if j['mts_idx'] == 1)
    assert reg > 0 and ts > 0, (reg, ts)
    # the threshold itself: 8204 (regular) / 8210 (transform skip) is the first isolated level through the limited prefix
    for lv, j, (lw, lh, mts, fam, v) in zip(levels, jobs, recs):
        if fam == 'isolated' and v in (8203, 8204, 8209, 8210):
            assert limited_prefix(lv, mts) == (v >= (8210 if mts == 1 else 8204)), (lw, lh, mts, v)
    # budget exhaustion: every coded coefficient non-zero and large spends more than the 1.75 (regular) / 2 (transform skip) context-coded
    # bins per coefficient the budget allows, in every (shape, mts_idx) of the set
    full = {r[:3] for lv, r in zip(levels, recs) if r[3] == 'max' and np.count_nonzero(lv) == min(lv.shape[0], 32) * min(lv.shape[1], 32)}
    assert full == {r[:3] for r in recs}


# ---- GPU tier -----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def eng8():
    with vb.IntraCostEngine(device=0, bit_depth=8, ctu_size=128) as e:
        yield e


@pytest.fixture(scope='module')
def eng9():
    with vb.IntraCostEngine(device=0, bit_depth=9, ctu_size=128) as e:
        yield e


@pytest.fixture(scope='module')
def eng10():
    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=128) as e:
        yield e


@pytest.fixture
def engines(request):
    return lambda bd: request.getfixturevalue('eng%d' % bd)


@pytest.mark.gpu
@pytest.mark.parametrize('chain', ('scalar', 'dq', 'rdoq'))
@pytest.mark.parametrize('bd', BDS)
def test_tu_chain_over_the_whole_qp_range(bd, chain, engines):
    """scalar quantiser with every mts_idx (incl. transform skip), dependent quantiser with MTS and LFNST 1 / 2 over all four LFNST sets,
    transform-skip RDOQ: every shape x family, corner shapes x family x every QP, lambda x1/4 x1 x4, VVCB_TU_RATE on every job"""
    eng = engines(bd)
    rng = np.random.default_rng(1000 * bd + ('scalar', 'dq', 'rdoq').index(chain))
    orig, jobs, resi, pred, rates, states, items = tu_cases(rng, bd, chain)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates, states=states)
    exp = ORACLE_CHAIN[chain](items, bd)
    assert_same(out, exp, items)
    assert_reach(reach(items, exp, bd, chain), bd, chain)
    assert eng.residual_bits(jobs, out['level'], states).tolist() == out['results']['frac_bits'].tolist()


@pytest.mark.gpu
def test_residual_bits_on_extreme_levels(eng10):
    """vvcb_residual_bits on level blocks of +-32767 / -32768, every coefficient non-zero, and isolated levels either side of the
    limited prefix, every shape x mts_idx (regular, MTS and transform-skip residual coding) against the oracle"""
    rng = np.random.default_rng(77)
    jobs, levels, states, recs, exp = level_cases(rng)
    got = eng10.residual_bits(jobs, np.concatenate([lv.ravel() for lv in levels]), states)
    bad = [(r, int(g), e) for r, g, e in zip(recs, got, exp) if int(g) != e]
    assert not bad, (len(bad), bad[:5])
    assert_level_reach(levels, jobs, recs)


@pytest.mark.gpu
@pytest.mark.parametrize('bd', BDS)
def test_range_refusals(bd, engines):
    """internal QP above 63 + 6 (bitDepth - 8), a lambda that is not finite, levels outside 16 bits"""
    eng = engines(bd)
    eng.frame_begin(np.zeros((64, 64), np.int16))
    z = np.zeros(16, np.int16)
    rates, states = np.zeros(1, vb.DQ_RATES_DTYPE), np.zeros(1, vb.CTX_STATES_DTYPE)
    top = max_qp(bd)
    for flags, mts in ((vb.TU_QUANT, 0), (vb.TU_QUANT | vb.TU_DEPQUANT, 0), (vb.TU_QUANT | vb.TU_RDOQ_TS, 1)):
        j = np.zeros(1, vb.TU_JOB_DTYPE)
        j['log2w'], j['log2h'], j['mts_idx'], j['flags'], j['lambda'] = 2, 2, mts, flags, 10.0
        j['qp_per'], j['qp_rem'] = top // 6, top % 6
        eng.tu_eval(j, z, z, rates=rates, states=states)                      # the top QP is accepted
        for per, rem in ((top // 6, top % 6 + 1) if top % 6 < 5 else (top // 6 + 1, 0), (top // 6 + 1, top % 6)):
            b = j.copy()
            b['qp_per'], b['qp_rem'] = per, rem
            with pytest.raises(vb.EngineError, match='malformed'):
                eng.tu_eval(b, z, z, rates=rates, states=states)
        if flags != vb.TU_QUANT:
            for lam in (np.inf, np.nan, -np.inf, 0.0):
                b = j.copy()
                b['lambda'] = lam
                with pytest.raises(vb.EngineError, match='malformed'):
                    eng.tu_eval(b, z, z, rates=rates, states=states)
    j = np.zeros(1, vb.TU_JOB_DTYPE)
    j['log2w'], j['log2h'] = 2, 2
    lv = np.zeros(16, np.int32)
    for v in (32767, -32768):
        lv[5] = v
        assert eng.residual_bits(j, lv, states)[0] > 0
    for v in (32768, -32769, 65535, -(1 << 31)):
        lv[5] = v
        with pytest.raises(vb.EngineError, match='malformed'):
            eng.residual_bits(j, lv, states)


# ---- CPU tier: the kernel source on host threads ------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def emul():
    import ctypes as C
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    subprocess.check_call(['make', '-s', '-f', 'tests/host_emul/Makefile'], cwd=root)
    return C.CDLL(os.path.join(root, 'tests/host_emul/libemul_rmd.so'))


@pytest.mark.parametrize('chain', ('scalar', 'dq', 'rdoq'))
@pytest.mark.parametrize('bd', BDS)
def test_emulated_tu_chain_at_the_range_limits(emul, bd, chain):
    """the corner shapes x every family at QPs 0, 1, 5, 6, 11, 12, 51 + QpBdOffset and the top QP"""
    rng = np.random.default_rng(2000 * bd + ('scalar', 'dq', 'rdoq').index(chain))
    top = max_qp(bd)
    orig, jobs, resi, pred, rates, states, items = tu_cases(rng, bd, chain, corner_qps=[0, 1, 5, 6, 11, 12, top - 12, top], sweep=False)
    out = run_emul_tu(emul, orig, bd, jobs, resi, pred, rates, states)
    exp = ORACLE_CHAIN[chain](items, bd)
    assert_same(out, exp, items)
    assert_reach(reach(items, exp, bd, chain), bd, chain, all_qps=False)


def test_emulated_residual_bits_on_extreme_levels(emul):
    rng = np.random.default_rng(78)
    jobs, levels, states, recs, exp = level_cases(rng)
    got = run_emul_rate(emul, jobs, np.concatenate([lv.ravel() for lv in levels]), states)
    bad = [(r, int(g), e) for r, g, e in zip(recs, got, exp) if int(g) != e]
    assert not bad, (len(bad), bad[:5])
    assert_level_reach(levels, jobs, recs)


def test_qp_list_and_shift_replica():
    """the QP list holds every boundary.  Over every shape x internal QP x lambda x1/4 .. x4 the dq_init_quant replica finds shift counts
    of 64 to 73 (on 4x4 blocks from signalled QP 48 on at the reference lambda, on larger blocks at higher QPs), and for every one of them
    f * 2^(count - 64) + .5 truncates to 0: the device shift (0) and the x86 one (count & 63) give the same distStepAdd."""
    for bd in BDS:
        q = qp_list(bd)
        assert {0, 1, 5, 6, 11, 12, 51 + 6 * (bd - 8), max_qp(bd)} <= set(q) and max(q) == max_qp(bd)
        assert all(6 * k - 1 in q and 6 * k in q for k in range(1, max_qp(bd) // 6 + 1))
        hits, worst = [], 0.0
        for lw, lh in SHAPES:
            for qp in range(max_qp(bd) + 1):
                for s in LAMBDA_SCALES:
                    d = dq_init_quant(bd, lw, lh, qp, ref_lambda(qp, s))
                    assert d['count'] <= 73
                    if d['count'] >= 64:
                        hits.append((lw, lh, qp, s))
                        worst = max(worst, d['f'] * float(1 << (d['count'] & 63)))
        assert min(qp for lw, lh, qp, s in hits if lw == lh == 2 and s == 1.0) == 48 + 6 * (bd - 8)
        assert worst < 0.5, worst
