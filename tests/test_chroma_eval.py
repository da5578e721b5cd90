"""Chroma intra candidates (vvcb_chroma_eval): Cb and Cr predicted under the 8 candidates of PU::getIntraChromaCandModes, with SAD and SATD.

The checker is oracle/vvc_oracle_chroma.c, restated from H.266 and the reference lines it cites; nothing here compares with the reference
encoder's own chroma output.  What ties it down: the kernel source (on host threads) and the device equal the oracle bit for bit; the
oracle's CCLM padding and sample-position rules are checked against hand computations; and the modes that chroma and luma compute
identically equal the pinned luma rough-mode-decision path (GPU)."""
import ctypes as C
import os
import subprocess
import sys
import time
import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LM, MDLM_L, MDLM_T, DM = 67, 68, 69, 70
CTU = 64                                   # luma CTU: chroma CTU rows start at multiples of 32


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


@pytest.fixture(scope='module')
def orc():
    subprocess.check_call(['make', '-s', '-f', 'tests/chroma_oracle/Makefile'], cwd=ROOT)
    L = C.CDLL(os.path.join(ROOT, 'tests/chroma_oracle/libchroma_oracle.so'))
    L.orc_chroma_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    L.orc_cclm_luma.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    L.orc_cclm_params.argtypes = [C.c_int] * 9 + [C.c_void_p] * 4 + [C.POINTER(C.c_int)] * 3
    return L


@pytest.fixture(scope='module')
def emul(tmp_path_factory):
    out = tmp_path_factory.mktemp('emul_chroma') / 'libemul_chroma.so'
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-g', '-ffp-contract=off', '-fPIC', '-shared', '-pthread', '-Wall', '-Wno-unused-function',
                           '-Wno-unknown-pragmas', '-Wno-unused-variable', '-o', str(out), os.path.join(ROOT, 'tests/host_emul/emul_chroma.cpp')])
    L = C.CDLL(str(out))
    L.emul_chroma_eval.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
    return L


def E():
    import vvc_intra_b200.engine as eng
    return eng


class Frame:
    """chroma planes Cb / Cr (original, reconstruction) of cw x ch and the luma reconstruction of 2cw x 2ch"""

    def __init__(self, rng, bd, cw, ch, kind):
        mx = (1 << bd) - 1

        def plane(h, w):
            if kind == 'flat':
                return np.full((h, w), int(rng.integers(0, mx + 1)), np.int16)
            if kind == 'checker':
                return (((np.arange(h)[:, None] + np.arange(w)[None, :]) & 1) * mx).astype(np.int16)
            return rng.integers(0, mx + 1, (h, w)).astype(np.int16)
        self.bd, self.cw, self.ch = bd, cw, ch
        self.cb, self.cr, self.cb_reco, self.cr_reco = (plane(ch, cw) for _ in range(4))
        self.luma = plane(2 * ch, 2 * cw)
        if kind == 'checker':
            self.cb_reco = (mx - self.cb_reco).astype(np.int16)
            self.luma[::2] = (mx - self.luma[::2]).astype(np.int16)

    def planes(self):
        self._keep = [np.ascontiguousarray(a) for a in (self.cb, self.cr, self.cb_reco, self.cr_reco)]
        return (C.c_void_p * 4)(*[a.ctypes.data for a in self._keep])


def visit(x, y, w, h, av, dm, cclm):
    v = np.zeros(1, E().CHROMA_VISIT_DTYPE)[0]
    v['x'], v['y'], v['log2w'], v['log2h'] = x, y, w.bit_length() - 1, h.bit_length() - 1
    v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = av
    v['dm_mode'], v['cclm'] = dm, cclm
    return v


SHAPES = [(1 << a, 1 << b) for a in range(2, 6) for b in range(2, 6)]
DMS = (0, 1, 18, 50, 66, 2, 34, 10, 27, 45, 60, 3)


def crossings(w, h, rng):
    """(x, y, availability) placements of a w x h chroma CU in a 160 x 128 chroma picture: none, all, partial above-right and below-left,
    the top-left alone, one side, a partial side, the picture's left and top edges, a CTU's first row and not"""
    uw, uh = w // 2, h // 2
    r = lambda n: int(rng.integers(0, n + 1))
    return [(64, 40, (0, 0, 0, 0, 0)), (64, 40, (1, uw, uw, uh, uh)), (64, 64, (1, uw, uw, uh, uh)),     # y = 64: a chroma CTU's first row
            (64, 40, (1, uw, r(uw), uh, r(uh))), (64, 64, (1, uw, r(uw), uh, r(uh))),
            (64, 40, (1, 0, 0, 0, 0)), (64, 40, (0, uw, r(uw), 0, 0)), (64, 40, (0, 0, 0, uh, r(uh))),
            (64, 40, (1, r(uw - 1), 0, uh, r(uh))), (64, 40, (1, uw, r(uw), r(uh - 1), 0)),
            (0, 40, (0, uw, r(uw), 0, 0)), (64, 0, (0, 0, 0, uh, r(uh))), (0, 0, (0, 0, 0, 0, 0))]


def make_visits(rng):
    out, k = [], 0
    for w, h in SHAPES:
        for x, y, av in crossings(w, h, rng):
            for cclm in (0, 1):
                out.append(visit(x, y, w, h, av, DMS[k % len(DMS)], cclm))
                k += 1
    return np.array(out, E().CHROMA_VISIT_DTYPE)


def oracle(orc, fr, visits, ctu=CTU, want_pred=True):
    res = np.zeros(len(visits), E().CHROMA_RESULT_DTYPE)
    total = sum(16 << (int(v['log2w']) + int(v['log2h'])) for v in visits)
    pred = np.zeros(total, np.int16) if want_pred else None
    luma = np.ascontiguousarray(fr.luma)
    orc.orc_chroma_batch(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, _p(visits), len(visits), _p(res), _p(pred) if want_pred else None)
    return res, pred


def emulate(emul, fr, visits, ctu=CTU):
    res = np.zeros(len(visits), E().CHROMA_RESULT_DTYPE)
    pred = np.zeros(sum(16 << (int(v['log2w']) + int(v['log2h'])) for v in visits), np.int16)
    luma = np.ascontiguousarray(fr.luma)
    emul.emul_chroma_eval(fr.planes(), fr.cw, _p(luma), luma.shape[1], fr.bd, ctu, _p(visits), len(visits), _p(pred), _p(res))
    return res, pred


# ---------------------------------------------------------------------------------------------------------------------------------
# the ABI
# ---------------------------------------------------------------------------------------------------------------------------------
def test_struct_sizes_match_the_header(tmp_path):
    src = tmp_path / 'sz.c'
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "vvc_intra_b200.h"\nint main(void){printf("%zu %zu %zu %zu\\n", sizeof(vvcb_chroma_visit), '
                   'sizeof(vvcb_chroma_result), offsetof(vvcb_chroma_result, sad), offsetof(vvcb_chroma_visit, dm_mode));return 0;}\n')
    exe = tmp_path / 'sz'
    subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), '-o', str(exe), str(src)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    eng = E()
    assert got == [eng.CHROMA_VISIT_DTYPE.itemsize, eng.CHROMA_RESULT_DTYPE.itemsize, eng.CHROMA_RESULT_DTYPE.fields['sad'][1],
                   eng.CHROMA_VISIT_DTYPE.fields['dm_mode'][1]]


# ---------------------------------------------------------------------------------------------------------------------------------
# the kernel source on host threads against the oracle
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('bd', (8, 9, 10))
@pytest.mark.parametrize('kind', ('noise', 'flat', 'checker'))
def test_emulated_kernel_matches_oracle(orc, emul, bd, kind):
    """chroma_eval_kernel (the kernel source, compiled for host threads) equals the oracle -- mode codes, every prediction sample, SAD and
    SATD of Cb and Cr -- on every shape 4..32 x 4..32, with cclm 0 and 1, DM on each of the four regular candidates and elsewhere, and the
    availability crossings of crossings()"""
    rng = np.random.default_rng(100 * bd + len(kind))
    fr = Frame(rng, bd, 160, 128, kind)
    visits = make_visits(rng)
    ores, opred = oracle(orc, fr, visits)
    eres, epred = emulate(emul, fr, visits)
    bad = [i for i in range(len(visits)) if ores[i].tobytes() != eres[i].tobytes()]
    assert not bad, [(visits[i], ores[i], eres[i]) for i in bad[:2]]
    assert np.array_equal(opred, epred)
    assert all(ores[i]['sad'][4, 0] == 0xFFFFFFFF for i in range(len(visits)) if not visits[i]['cclm'])
    assert sum(int(v['cclm']) for v in visits) * 2 == len(visits) and len(visits) == 16 * 13 * 2


def test_candidate_list_substitutes_dm(orc):
    """PLANAR, VER, HOR, DC, LM, MDLM_L, MDLM_T, DM; the first of the four regular candidates equal to DM becomes VDIA (66)"""
    rng = np.random.default_rng(1)
    fr = Frame(rng, 10, 160, 128, 'noise')
    for dm, want in ((0, [66, 50, 18, 1]), (50, [0, 66, 18, 1]), (18, [0, 50, 66, 1]), (1, [0, 50, 18, 66]), (66, [0, 50, 18, 1]), (7, [0, 50, 18, 1])):
        res, _ = oracle(orc, fr, np.array([visit(64, 40, 8, 8, (1, 4, 0, 4, 0), dm, 1)], E().CHROMA_VISIT_DTYPE))
        assert res[0]['mode'].tolist() == want + [LM, MDLM_L, MDLM_T, DM]


# ---------------------------------------------------------------------------------------------------------------------------------
# oracle properties: CCLM rules against hand computations
# ---------------------------------------------------------------------------------------------------------------------------------
DIV_SIG = (0, 7, 6, 5, 5, 4, 4, 3, 3, 2, 2, 1, 1, 1, 1, 0)


def lm_from_samples(selY, selC, bd):
    """(a, k, b) from the four selected (luma, chroma) pairs: min/max grouping, averages, the DivSigTable division (H.266 CCLM clause)"""
    selY, selC = list(selY), list(selC)
    if len(selY) == 2:
        selY, selC = [selY[1], selY[0], selY[1], selY[0]], [selC[1], selC[0], selC[1], selC[0]]
    mn, mx = [0, 2], [1, 3]
    if selY[mn[0]] > selY[mn[1]]:
        mn = [mn[1], mn[0]]
    if selY[mx[0]] > selY[mx[1]]:
        mx = [mx[1], mx[0]]
    if selY[mn[0]] > selY[mx[1]]:
        mn, mx = mx, mn
    if selY[mn[1]] > selY[mx[0]]:
        mn[1], mx[0] = mx[0], mn[1]
    minY, minC = (selY[mn[0]] + selY[mn[1]] + 1) >> 1, (selC[mn[0]] + selC[mn[1]] + 1) >> 1
    maxY, maxC = (selY[mx[0]] + selY[mx[1]] + 1) >> 1, (selC[mx[0]] + selC[mx[1]] + 1) >> 1
    diff = maxY - minY
    if diff <= 0:
        return 0, 0, minC
    diffC = maxC - minC
    x = diff.bit_length() - 1
    nd = ((diff << 4) >> x) & 15
    v = DIV_SIG[nd] | 8
    x += nd != 0
    y = abs(diffC).bit_length()
    a = (diffC * v + ((1 << y) >> 1)) >> y
    k = 3 + x - y
    if k < 1:
        k, a = 1, (0 if a == 0 else (-15 if a < 0 else 15))
    return a, k, minC - ((a * minY) >> k)


def lm_pred(ds, a, k, b, bd):
    return np.clip(((ds.astype(np.int64) * a) >> k) + b, 0, (1 << bd) - 1)


def ds6(Y, r, c0, cl):
    """[1 2 1; 1 2 1] / 8 at luma rows r, r + 1: centre column c0, left column cl"""
    return (2 * int(Y[r, c0]) + int(Y[r, c0 + 1]) + int(Y[r, cl]) + 2 * int(Y[r + 1, c0]) + int(Y[r + 1, c0 + 1]) + int(Y[r + 1, cl]) + 4) >> 3


def one_visit(orc, fr, v, ctu=CTU):
    res, pred = oracle(orc, fr, np.array([v], E().CHROMA_VISIT_DTYPE), ctu)
    w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
    return res[0], pred.reshape(8, 2, h, w)


@pytest.mark.parametrize('bd', (8, 10))
def test_no_neighbours_predicts_mid_grey(orc, bd):
    rng = np.random.default_rng(bd)
    fr = Frame(rng, bd, 160, 128, 'noise')
    for w, h in SHAPES:
        _, pred = one_visit(orc, fr, visit(64, 40, w, h, (1, 0, 0, 0, 0), 5, 1))
        assert (pred[4:7] == 1 << (bd - 1)).all()


def test_flat_luma_neighbours_give_min_chroma(orc):
    """diff = 0 (every selected luma value equal): a = 0, k = 0, b = minC, the average of the chroma at the first min-group pair"""
    rng = np.random.default_rng(3)
    fr = Frame(rng, 10, 160, 128, 'noise')
    fr.luma[:, :] = 300
    for w, h in SHAPES:
        x, y = 64, 40
        _, pred = one_visit(orc, fr, visit(x, y, w, h, (1, w // 2, 0, h // 2, 0), 5, 1))
        top, left = fr.cb_reco[y - 1, x:x + w], fr.cb_reco[y:y + h, x - 1]
        minC = (int(top[w >> 2]) + int(left[h >> 2]) + 1) >> 1          # LM picks top w/4, 3w/4, left h/4, 3h/4; groups {0, 2} / {1, 3}
        assert (pred[4, 0] == minC).all(), (w, h)


@pytest.mark.parametrize('w,h', [(4, 4), (8, 8), (16, 8), (32, 4), (4, 32), (32, 32)])
def test_mdlm_t_without_above_right_picks_hand_positions(orc, w, h):
    """MDLM_T with n_above_right = 0: numSampT = w, numIs4N = 1, so startPos = w >> 3, pickStep = max(1, w >> 2), four positions"""
    rng = np.random.default_rng(w * h)
    fr = Frame(rng, 10, 160, 128, 'noise')
    x, y = 64, 40
    res, pred = one_visit(orc, fr, visit(x, y, w, h, (1, w // 2, 0, h // 2, h // 2), 5, 1))
    pos = [(w >> 3) + i * max(1, w >> 2) for i in range(4)]
    Y = fr.luma
    dsT = [ds6(Y, 2 * y - 2, 2 * (x + p), 2 * (x + p) - 1) for p in pos]
    selC = [int(fr.cb_reco[y - 1, x + p]) for p in pos]
    a, k, b = lm_from_samples(dsT, selC, 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - 1) for i in range(w)] for j in range(h)])
    assert np.array_equal(pred[6, 0], lm_pred(ds, a, k, b, 10))


def _padding_case(orc, w, h, av, mode, ctu=CTU, x=64, y=40, poison=None):
    """a 10-bit picture with strongly correlated luma / chroma (a != 0); poison(Y) marks luma samples a wrong padding would read"""
    rng = np.random.default_rng(w + 7 * h + mode)
    fr = Frame(rng, 10, 160, 128, 'noise')
    fr.luma = (rng.integers(0, 1024, (256, 320))).astype(np.int16)
    if poison:
        poison(fr.luma)
    cy = (fr.luma[1::2, 0::2].astype(np.int32) + 1) >> 1          # chroma follows the luma (odd rows, even columns: not the poisoned samples)
    fr.cb_reco, fr.cr_reco = cy.astype(np.int16), (1023 - cy).astype(np.int16)
    return fr, one_visit(orc, fr, visit(x, y, w, h, av, 5, 1), ctu)[1][mode - LM + 4]


def test_padding_block_without_left_uses_column_zero(orc):
    """no left neighbours: in the block, luma column -1 is replaced by column 0 (leftPadding); the poisoned column -1 must not matter"""
    w, h, x, y = 8, 8, 64, 40
    fr, pred = _padding_case(orc, w, h, (0, w // 2, w // 2, 0, 0), MDLM_T, poison=lambda Y: Y.__setitem__((slice(None), 2 * 64 - 1), 1023))
    Y = fr.luma
    dsT = [ds6(Y, 2 * y - 2, 2 * (x + p), 2 * (x + p) - (0 if p == 0 else 1)) for p in range(2 * w)]
    pos = [(2 * w >> 3) + i * max(1, 2 * w >> 2) for i in range(4)]
    a, k, b = lm_from_samples([dsT[p] for p in pos], [int(fr.cb_reco[y - 1, x + p]) for p in pos], 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - (0 if i == 0 else 1)) for i in range(w)] for j in range(h)])
    assert a != 0
    assert np.array_equal(pred[0], lm_pred(ds, a, k, b, 10))


def test_padding_top_without_left_uses_column_zero(orc):
    """no left neighbours: top neighbour 0 reads luma column 0 twice instead of column -1 (picked: MDLM_T of a 4-wide block takes 0..3)"""
    w, h, x, y = 4, 8, 64, 40
    fr, pred = _padding_case(orc, w, h, (0, 2, 0, 0, 0), MDLM_T, poison=lambda Y: Y.__setitem__((slice(2 * 40 - 2, 2 * 40), 2 * 64 - 1), 1023))
    Y = fr.luma
    dsT = [ds6(Y, 2 * y - 2, 2 * (x + p), 2 * (x + p) - (0 if p == 0 else 1)) for p in range(4)]
    a, k, b = lm_from_samples(dsT, [int(fr.cb_reco[y - 1, x + p]) for p in range(4)], 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - (0 if i == 0 else 1)) for i in range(w)] for j in range(h)])
    assert np.array_equal(pred[0], lm_pred(ds, a, k, b, 10))


def test_padding_top_with_left_reads_the_corner(orc):
    """left available: top neighbour 0 reads the luma above-left corner (column -1 of rows -2, -1), which differs from column 0 here"""
    w, h, x, y = 4, 8, 64, 40
    fr, pred = _padding_case(orc, w, h, (1, 2, 0, 4, 0), MDLM_T, poison=lambda Y: Y.__setitem__((slice(2 * 40 - 2, 2 * 40), 2 * 64 - 1), 1023))
    Y = fr.luma
    dsT = [ds6(Y, 2 * y - 2, 2 * (x + p), 2 * (x + p) - 1) for p in range(4)]
    a, k, b = lm_from_samples(dsT, [int(fr.cb_reco[y - 1, x + p]) for p in range(4)], 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - 1) for i in range(w)] for j in range(h)])
    assert np.array_equal(pred[0], lm_pred(ds, a, k, b, 10))


def test_padding_top_at_a_ctu_boundary_uses_one_row(orc):
    """the block's first chroma row starts a CTU: the top neighbours are [1 2 1] / 4 on luma row -1 alone; the poisoned row -2 must not
    matter (y = 32: chroma CTU rows of 32 with a 64-sample luma CTU)"""
    w, h, x, y = 4, 8, 64, 32
    fr, pred = _padding_case(orc, w, h, (1, 2, 0, 4, 0), MDLM_T, y=y, poison=lambda Y: Y.__setitem__((2 * 32 - 2, slice(None)), 1023))
    Y = fr.luma
    r = 2 * y - 1
    dsT = [(2 * int(Y[r, 2 * (x + p)]) + int(Y[r, 2 * (x + p) + 1]) + int(Y[r, 2 * (x + p) - 1]) + 2) >> 2 for p in range(4)]
    a, k, b = lm_from_samples(dsT, [int(fr.cb_reco[y - 1, x + p]) for p in range(4)], 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - 1) for i in range(w)] for j in range(h)])
    assert np.array_equal(pred[0], lm_pred(ds, a, k, b, 10))
    _, pred64 = _padding_case(orc, w, h, (1, 2, 0, 4, 0), MDLM_T, y=y, ctu=128, poison=lambda Y: Y.__setitem__((2 * 32 - 2, slice(None)), 1023))
    assert not np.array_equal(pred64[0], pred[0])                        # inside a 128 CTU the same block reads both rows


def test_padding_left_reads_three_columns(orc):
    """the left neighbours read luma columns -3..-1 of rows 2j, 2j + 1 (no padding); below-left ones with MDLM_L, four positions of a
    4-high block: 0..3"""
    w, h, x, y = 8, 4, 64, 40
    fr, pred = _padding_case(orc, w, h, (1, 4, 0, 2, 2), MDLM_L)
    Y = fr.luma
    dsL = [ds6(Y, 2 * (y + j), 2 * x - 2, 2 * x - 3) for j in range(h + min(4, w))]
    pos = [(h + 4 >> 3) + i * max(1, h + 4 >> 2) for i in range(4)]
    a, k, b = lm_from_samples([dsL[p] for p in pos], [int(fr.cb_reco[y + p, x - 1]) for p in pos], 10)
    ds = np.array([[ds6(Y, 2 * (y + j), 2 * (x + i), 2 * (x + i) - 1) for i in range(w)] for j in range(h)])
    assert a != 0
    assert np.array_equal(pred[0], lm_pred(ds, a, k, b, 10))


# ---------------------------------------------------------------------------------------------------------------------------------
# on the device
# ---------------------------------------------------------------------------------------------------------------------------------
def _engine(fr, ctu=CTU):
    import vvc_intra_b200 as vb
    eng = vb.IntraCostEngine(device=0, bit_depth=fr.bd, ctu_size=ctu)
    eng.frame_begin(np.zeros((2 * fr.ch, 2 * fr.cw), np.int16))
    eng.reco_update(fr.luma)
    eng.chroma_frame_begin(fr.cb, fr.cr)
    eng.chroma_reco_update(fr.cb_reco, fr.cr_reco)
    return eng


@pytest.mark.gpu
@pytest.mark.parametrize('bd', (8, 9, 10))
def test_device_matches_oracle_walk_and_large_batches(orc, bd):
    """the device equals the oracle bit for bit -- predictions, SAD, SATD -- on a walk-sized batch (~30 visits) and inside one of at least
    100 000 visits"""
    rng = np.random.default_rng(200 + bd)
    for kind in ('noise', 'checker'):
        fr = Frame(rng, bd, 160, 128, kind)
        visits = make_visits(rng)
        ores, opred = oracle(orc, fr, visits)
        with _engine(fr) as eng:
            walk = visits[rng.permutation(len(visits))[:30]]
            wres, wpred = oracle(orc, fr, walk)
            dres, dpred = eng.chroma_eval(walk, want_pred=True)
            assert dres.tobytes() == wres.tobytes()
            assert np.array_equal(np.concatenate([p.ravel() for p in dpred]), wpred)
            dres, dpred = eng.chroma_eval(visits, want_pred=True)
            assert dres.tobytes() == ores.tobytes()
            assert np.array_equal(np.concatenate([p.ravel() for p in dpred]), opred)
            reps = -(-100000 // len(visits))
            big = eng.chroma_eval(np.tile(visits, reps))
            assert len(big) >= 100000 and big.tobytes() == np.tile(ores, reps).tobytes()


def _luma_twin(v, eng_mod):
    """the luma visit whose availability equals the chroma visit's in samples (even chroma counts)"""
    lv = np.zeros(1, eng_mod.VISIT_DTYPE)[0]
    lv['x'], lv['y'], lv['log2w'], lv['log2h'] = v['x'], v['y'], v['log2w'], v['log2h']
    lv['avail_al'] = v['avail_al']
    for f in ('n_above', 'n_above_right', 'n_left', 'n_below_left'):
        assert v[f] % 2 == 0
        lv[f] = v[f] // 2
    lv['flags'] = 3
    lv['mpm'] = (0, 1, 50, 18, 46, 54)
    lv['num_mpm_cand'] = 1
    lv['sqrt_lambda'] = 10.0
    return lv


@pytest.mark.gpu
def test_modes_shared_with_luma_equal_the_pinned_luma_path(orc):
    """A chroma plane loaded as the picture of a luma context: DC, HOR and VER on every shape, planar where the luma path does not smooth
    (w * h <= 32) and the integer-slope modes whose luma parameters have no smoothing predict the same samples with the same SAD and SATD
    on both paths (vvcb_rmd_pred, vvcb_rmd_detail)"""
    import vvc_intra_b200 as vb
    eng_mod = E()
    rng = np.random.default_rng(77)
    fr = Frame(rng, 10, 160, 128, 'noise')
    P = orc                                                               # holds the oracle's orc_ipa_init too

    class Ipa(C.Structure):
        _fields_ = [(n, C.c_int) for n in ('is_ver', 'mrl', 'ref_filter', 'interp', 'pdpc', 'angle', 'inv_angle', 'ang_scale')]
    P.orc_ipa_init.argtypes = [C.c_int] * 5 + [C.POINTER(Ipa)]
    cases = []
    for w, h in SHAPES:
        modes = [1, 18, 50] + ([0] if w * h <= 32 else [])
        for m in range(2, 67):
            p = Ipa()
            P.orc_ipa_init(w, h, m, 0, 0, C.byref(p))
            if p.angle and p.angle % 32 == 0 and not p.ref_filter:
                modes.append(m)
        for av in ((1, w // 2, w // 2, h // 2, h // 2), (0, w // 2, 0, 0, 0), (1, 0, 0, h // 2, 0), (0, 0, 0, 0, 0)):
            av = tuple(a - a % 2 if i else a for i, a in enumerate(av))
            for m in modes:
                cases.append((visit(64, 40, w, h, av, m, 0), m))
    assert any(m == 2 for _, m in cases) and any(m == 66 for _, m in cases) and any(m == 34 for _, m in cases)
    visits = np.array([c[0] for c in cases], eng_mod.CHROMA_VISIT_DTYPE)
    with _engine(fr) as eng:
        cres, cpred = eng.chroma_eval(visits, want_pred=True)
    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=CTU) as leng:
        leng.frame_begin(fr.cb)
        leng.reco_update(fr.cb_reco)
        lv = np.array([_luma_twin(v, eng_mod) for v in visits], eng_mod.VISIT_DTYPE)
        _, det = leng.rmd_eval(lv, detail=True)
        compared = 0
        for i, (v, m) in enumerate(cases):
            slot = 7                                                      # DM
            lp = leng.rmd_pred(lv[i], m)
            assert np.array_equal(cpred[i][slot, 0], lp), (v, m)
            if det[i]['sad'][m] != 0xFFFFFFFF:
                assert (cres[i]['sad'][slot, 0], cres[i]['satd'][slot, 0]) == (det[i]['sad'][m], det[i]['satd'][m]), (v, m)
                compared += 1
    assert compared > len(cases) // 2


def sweep_visits(rng, cw=960, ch=540):
    """every aligned 4..32 chroma block of a 1080p 4:2:0 picture, availability from its position"""
    out = []
    for w, h in SHAPES:
        for y in range(0, ch - h + 1, h):
            for x in range(0, cw - w + 1, w):
                nl = h // 2 if x else 0
                na = w // 2 if y else 0
                nar = min(w // 2, (cw - x - w) // 2) if y else 0
                nbl = min(h // 2, (ch - y - h) // 2) if x else 0
                out.append((x, y, w.bit_length() - 1, h.bit_length() - 1, int(x > 0 and y > 0), na, nar, nl, nbl))
    v = np.zeros(len(out), E().CHROMA_VISIT_DTYPE)
    a = np.array(out)
    for i, f in enumerate(('x', 'y', 'log2w', 'log2h', 'avail_al', 'n_above', 'n_above_right', 'n_left', 'n_below_left')):
        v[f] = a[:, i]
    v['dm_mode'] = rng.integers(0, 67, len(v))
    v['cclm'] = 1
    return v


@pytest.mark.gpu
def test_1080p_sweep_is_deterministic_and_matches_the_oracle(orc):
    rng = np.random.default_rng(1080)
    fr = Frame(rng, 10, 960, 540, 'noise')
    visits = sweep_visits(rng)
    with _engine(fr) as eng:
        r1 = eng.chroma_eval(visits)
        r2 = eng.chroma_eval(visits)
    assert r1.tobytes() == r2.tobytes()
    pick = rng.choice(len(visits), 2000, replace=False)
    ores, _ = oracle(orc, fr, visits[pick], want_pred=False)
    assert r1[pick].tobytes() == ores.tobytes()


@pytest.mark.gpu
def test_refusals(tmp_path):
    """every refusal of the chroma entry points, and the broker proxy's"""
    import vvc_intra_b200 as vb
    rng = np.random.default_rng(9)
    fr = Frame(rng, 10, 160, 128, 'noise')
    good = visit(64, 40, 8, 8, (1, 4, 4, 4, 4), 5, 1)
    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=CTU) as eng:
        with pytest.raises(vb.engine.EngineError):
            eng.chroma_frame_begin(fr.cb, fr.cr)                          # before vvcb_frame_begin
        eng.frame_begin(np.zeros((256, 320), np.int16))
        with pytest.raises(vb.engine.EngineError):
            eng.chroma_eval(np.array([good]))                             # before vvcb_chroma_frame_begin
        with pytest.raises(vb.engine.EngineError):
            eng.chroma_reco_update(fr.cb_reco, fr.cr_reco)
        with pytest.raises(vb.engine.EngineError):
            eng.chroma_frame_begin(fr.cb[:, :80], fr.cr[:, :80])          # not half the luma size
        eng.chroma_frame_begin(fr.cb, fr.cr)
        with pytest.raises(vb.engine.EngineError):
            eng.chroma_reco_update(fr.cb_reco[:, :8], fr.cr_reco[:, :8], x=156)
        eng.chroma_eval(np.array([good]))
        bad = []
        for f, val in (('log2w', 1), ('log2h', 1), ('log2w', 6), ('log2h', 6), ('n_above', 5), ('n_above_right', 5), ('n_left', 5),
                       ('n_below_left', 5), ('avail_al', 2), ('dm_mode', 67), ('cclm', 2), ('x', 156), ('y', 124), ('x', -2), ('x', 63), ('y', 41)):
            b = good.copy()
            b[f] = val
            bad.append(b)
        for f, x, y in (('n_left', 0, 40), ('n_above', 64, 0), ('avail_al', 0, 40), ('n_above_right', 146, 40), ('n_below_left', 64, 114)):
            b = good.copy()
            b['x'], b['y'] = x, y
            for g in ('avail_al', 'n_above', 'n_above_right', 'n_left', 'n_below_left'):
                b[g] = 0
            b[f] = 1 if f == 'avail_al' else 4
            bad.append(b)
        for b in bad:
            with pytest.raises(vb.engine.EngineError):
                eng.chroma_eval(np.array([good, b]))
    # through the broker: the proxy context refuses every chroma entry point
    root = ROOT
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([os.path.join(root, 'vvc_intra_b200/vvcb_broker'), path, '--bit-depth', '10', '--ctu', str(CTU), '--clients', '2',
                               '--frame', '320x256', '--workers', '1'], env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        code = ('import numpy as np, vvc_intra_b200 as vb\n'
                'from vvc_intra_b200 import engine as E\n'
                'eng = vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=%d)\n'
                'eng.frame_begin(np.zeros((256, 320), np.int16))\n'
                'out = []\n'
                'for f in (lambda: eng.chroma_frame_begin(np.zeros((128, 160), np.int16), np.zeros((128, 160), np.int16)),\n'
                '          lambda: eng.chroma_reco_update(np.zeros((8, 8), np.int16), np.zeros((8, 8), np.int16)),\n'
                '          lambda: eng.chroma_eval(np.zeros(1, E.CHROMA_VISIT_DTYPE))):\n'
                '    try:\n'
                '        f(); out.append("accepted")\n'
                '    except E.EngineError as e:\n'
                '        out.append("broker" in str(e))\n'
                'print(out)\n') % CTU
        r = None
        for _ in range(100):                                              # the server creates the broker file when it is ready
            if os.path.exists(path):
                r = subprocess.run([sys.executable, '-c', code], cwd=root, env=dict(env0, VVCB_BROKER=path), stdout=subprocess.PIPE,
                                   stderr=subprocess.STDOUT, text=True, timeout=300)
                break
            time.sleep(0.2)
        assert r is not None and r.returncode == 0, r and r.stdout[-2000:]
        assert r.stdout.strip().splitlines()[-1] == '[True, True, True]', r.stdout[-2000:]
    finally:
        subprocess.run([os.path.join(root, 'vvc_intra_b200/vvcb_broker'), path, '--stop'], env=env0, timeout=60)
        try:
            server.wait(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
            server.wait()
