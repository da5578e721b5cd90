"""CPU tests: the plain-C oracle (oracle/vvc_oracle.c) against records captured from the UNMODIFIED
reference encoder (tests/golden/*.bin.gz, made by tools/make_golden.py).  This is what pins the oracle."""
import numpy as np
import pytest

from oracle import oracle_py as O
import golden_util as G

FIXTURES = ['ref_8b_128x64_qp32', 'ref_10b_192x128_qp27']


@pytest.mark.parametrize('name', FIXTURES)
def test_fixture_covers_all_shapes(name):
    visits, _ = G.load_fixture(name)
    shapes = {(v['head']['w'], v['head']['h']) for v in visits}
    want = {(w, h) for w in (4, 8, 16, 32) for h in (4, 8, 16, 32)} | {(64, 64)}
    assert want <= shapes


@pytest.mark.parametrize('name', FIXTURES)
def test_reference_lines(name):
    """a1-a3: xFillReferenceSamples / xFilterReferenceSamples for lines 0, 1 and 3."""
    visits, _ = G.load_fixture(name)
    n = 0
    for v in visits:
        hd = v['head']
        w, h, bd = hd['w'], hd['h'], hd['bd']
        for r in v['refs']:
            reco = np.zeros((2 * h + 8, 2 * w + 8), np.int16)
            reco[0:4, :] = r['reco_top']
            reco[4:, 0:4] = r['reco_left']
            top, left = O.ref_fill(reco, 4, 4, w, h, r['mrl'], bd, r['avail_al'], r['n_above'], r['n_above_right'],
                                   r['n_left'], r['n_below_left'])
            assert np.array_equal(top, r['unf_top']) and np.array_equal(left, r['unf_left'])
            if r['has_filt']:
                ft, fl = O.ref_filter(r['unf_top'], r['unf_left'], w, h, r['mrl'])
                assert np.array_equal(ft, r['filt_top']) and np.array_equal(fl, r['filt_left'])
            n += 1
    assert n > 100


@pytest.mark.parametrize('name', FIXTURES)
def test_prediction_distortion_and_bits(name):
    """a4-a8, a10: parameters, prediction samples, SAD, SATD and mode bits of every recorded evaluation."""
    visits, _ = G.load_fixture(name)
    n_pred = n_full = 0
    for v in visits:
        hd = v['head']
        w, h, bd = hd['w'], hd['h'], hd['bd']
        for e in v['evals']:
            r = v['refs'][e['ref_idx']]
            if e['mip']:
                pred = O.pred_mip(r['unf_top'], r['unf_left'], w, h, bd, e['mode'])
            else:
                ipa = O.ipa_init(w, h, e['mode'], e['mrl'])
                if e['mode'] > 1:
                    assert (ipa.is_ver, ipa.angle, ipa.inv_angle) == (e['is_ver'], e['angle'], e['inv_angle'])
                    if e['pdpc'] and e['angle'] > 0:
                        assert ipa.ang_scale == e['ang_scale']
                assert (ipa.ref_filter, ipa.interp, ipa.pdpc) == (e['ref_filter'], e['interp'], e['pdpc'])
                src = (r['filt_top'], r['filt_left']) if ipa.ref_filter else (r['unf_top'], r['unf_left'])
                pred = O.pred_regular(src[0], src[1], w, h, bd, e['mode'], ipa)
            assert O.fnv1a(pred) == e['hash'], (w, h, e['mip'], e['mrl'], e['mode'])
            if 'pred' in e:
                assert np.array_equal(pred, e['pred'])
                n_full += 1
            assert O.sad(hd['org'], pred) == e['sad']
            assert O.satd(hd['org'], pred) == e['satd']
            if 'bits' in e:
                got = O.mode_bits(hd['rates'], hd['mpm'], w, h, (hd['y'] & 127) != 0, 1, e['mip'], e['mrl'], e['mode'])
                assert got == e['bits']
            n_pred += 1
    assert n_pred > 2000
    if name == 'ref_8b_128x64_qp32':
        assert n_full > 500


@pytest.mark.parametrize('name', FIXTURES)
def test_rmd_visit_lists(name):
    """a9: whole visits from the reco window to the candidate lists (costs compared as exact doubles)."""
    visits, _ = G.load_fixture(name)
    orig, reco, arr = G.build_atlas(visits)
    bd = visits[0]['head']['bd']
    res, det = O.rmd_batch(orig, reco, bd, 128, arr)
    errs = []
    for v, r, d in zip(visits, res, det):
        errs += G.check_visit_against_reference(v, r, d)
    assert not errs, errs[:5]


def test_satd_normalisation_shortcut_is_exact():
    """The CUDA kernel replaces (int)(s / sqrt(N) * 2) (CL/RdCost.cpp:2452,2662) by one multiply with a
    reciprocal; prove it over the whole reachable range of s.  By Parseval the sum of the 128 absolute Hadamard coefficients of a
    16x8 tile is at most 128 * sqrt(128) * max|residual|: < 1.5e6 for 10-bit residuals, < 6e6 even for 12-bit ones."""
    s = np.arange(0, 1 << 23, dtype=np.int64)
    for n in (128.0, 32.0):
        ref = (s / np.sqrt(n) * 2).astype(np.int64)
        c = np.float64(2.0) / np.sqrt(np.float64(n))
        fast = (s.astype(np.float64) * c).astype(np.int64)
        assert np.array_equal(ref, fast)


def test_mpm_derivation_matches_recorded_lists():
    """PU::getIntraMPMs restatement: every recorded MPM list must be reachable from some (left, above) pair."""
    table = {}
    for L in range(67):
        for A in range(67):
            m, n = O.intra_mpms(L, A)
            table[tuple(m)] = n
    for name in FIXTURES:
        visits, _ = G.load_fixture(name)
        for v in visits:
            key = tuple(int(x) for x in v['head']['mpm'])
            assert key in table
