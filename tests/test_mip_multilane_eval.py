"""MIP slots of two or more lanes (every MIP shape above 8x8 but the 4x4 / 8x4 / 4x8 / 8x8 ones a lane owns): the evaluation kernels
predict them in registers, each lane computing the reduced samples under its unit plus the border its up-sampling reads.  A wrong border
(the neighbouring unit's reduced sample, or the boundary sample, taken for the other) shows here, against the oracle byte for byte:
SAD / SATD detail tables, result records and prediction samples of every MIP mode in both orientations, at bit depths 8 and 10.

Reconstruction and original are seeded noise over the whole sample range, so the reduced samples of neighbouring units differ from each
other and from the boundary sample at the same position; the case set asserts that from a numpy replica of the MIP matrix product.

Item flavours: sweep-sized calls (packed items for 16x4, 4x16, 16x8, 8x16; plain items for the larger shapes), walk-sized calls (one
launch for every bucket, rmd_eval_any_kernel) and the prediction-output kernels.  CPU tier: the kernel source on host threads
(tests/host_emul); GPU tier: the library (the IDP.2A branches of the matrix product are device-only)."""
import ctypes as C
import functools
import os
import subprocess

import numpy as np
import pytest

import vvc_intra_b200 as vb
from oracle import oracle_py as O
from test_rmd_range_limits import mip_family, mip_num_modes, random_visit_fields, rom_tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BDS = (8, 10)
# (w, h) of every MIP shape whose slots span two or more lanes
SHAPES = [(16, 4), (4, 16), (16, 8), (8, 16), (16, 16), (32, 8), (8, 32), (32, 16), (16, 32), (32, 32),
          (64, 16), (16, 64), (64, 32), (32, 64), (64, 64)]
PER_SHAPE = 8
CTU = 128


# ---- the cases -------------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def case(bd):
    """PER_SHAPE visits of every shape on a noise picture, all lines available, MIP enabled; one visit per shape at x = 0 or y = 0"""
    rng = np.random.default_rng(4242 + bd)
    H, W = 640, 1024
    reco = rng.integers(0, 1 << bd, (H, W)).astype(np.int16)
    orig = rng.integers(0, 1 << bd, (H, W)).astype(np.int16)
    visits = np.zeros(len(SHAPES) * PER_SHAPE, O.VISIT_DTYPE)
    i = 0
    for s, (w, h) in enumerate(SHAPES):
        for j in range(PER_SHAPE):
            v = visits[i]
            random_visit_fields(v, rng, w, h)
            v['log2w'], v['log2h'] = w.bit_length() - 1, h.bit_length() - 1
            v['x'] = 0 if j == 0 else 64 + 8 * int(rng.integers(0, (W - 192) // 8))
            v['y'] = 0 if j == 1 else 64 + 8 * int(rng.integers(0, (H - 192) // 8))
            v['avail_al'] = int(v['x'] > 0 and v['y'] > 0)
            v['n_above'], v['n_above_right'] = (w // 4, w // 4) if v['y'] > 0 else (0, 0)
            v['n_left'], v['n_below_left'] = (h // 4, h // 4) if v['x'] > 0 else (0, 0)
            v['flags'] = 1 if 64 in (w, h) and w != h else 0    # MIP on; MRL as the position allows, but not for 64x16 ... 32x64, whose
                                                                  # line buffers hold a 64-sample side on reference line 0 only
            i += 1
    ora, odet = O.rmd_batch(orig, reco, bd, CTU, visits)
    return orig, reco, visits, ora, odet


def mip_reduced(top, left, w, h, bd, mode):
    """reduced prediction (redH x redW, block orientation, clipped) of one MIP mode: CL/MatrixIntraPrediction.cpp:71-124, 637-741"""
    T = rom_tables()
    fam, n = mip_family(w, h), mip_num_modes(w, h)
    small = fam < 2
    bsz = 4 if (w > 4 or h > 4) else 2
    redW, redH = (4, 4) if small else (min(w, 8), min(h, 8))
    name = ('4x4', '8x8', '16x16')[fam]
    mats, shifts, offs = T['kMipMatrix' + name], T['kMipShift' + name], T['kMipOffset' + name]
    rows_, cols = (16, 16, 64)[fam], (4, 8, 7)[fam]

    def down(src):
        f = len(src) // bsz
        s = src.reshape(bsz, f).sum(1)
        return s if f == 1 else (s + (f >> 1)) >> (f.bit_length() - 1)
    bT, bL = down(top[1:w + 1].astype(np.int64)), down(left[1:h + 1].astype(np.int64))
    t = 1 if mode > n // 2 else 0
    widx = mode - n // 2 if t else mode
    inp = np.concatenate([bL, bT] if t else [bT, bL])
    first = int(inp[0])
    inp[1:] -= first
    inp[0] = first - (1 << (bd - 1)) if small else 0
    lho, lvo = (w == 4 and h >= 16), (h == 4 and w >= 16)
    iw, ih = (redH, redW) if t else (redW, redH)
    if t:
        lho, lvo = lvo, lho
    yy, xx = np.mgrid[0:ih, 0:iw]
    rows = ((2 * yy if lvo else yy) * (iw if small else 8) + (2 * xx if lho else xx)).ravel()
    M = mats[widx * rows_ * cols:(widx + 1) * rows_ * cols].reshape(rows_, cols)[rows]
    acc = M @ (inp if small else inp[1:])
    off = (1 << (int(shifts[widx]) - 1)) - int(offs[widx]) * int(inp.sum())
    v = np.clip(((acc + off) >> int(shifts[widx])) + first, 0, (1 << bd) - 1).reshape(ih, iw)
    return v.T if t else v


def unit_borders(w, h):
    """for each reduced position: does a unit border of the evaluation kernels run between it and its left / upper neighbour"""
    redW, redH = min(w, 8), min(h, 8)
    upH, upV = w // redW, h // redH
    S = 4 if min(w, h) == 4 else 8
    # a lane's piece is 4 rows x 4 (S = 4) or 8 columns: a border lies between reduced samples that fall into different pieces
    pw, ph = (4, 4) if S == 4 else (8, 4)
    colB = np.array([rx > 0 and (rx * upH) // pw != ((rx - 1) * upH) // pw for rx in range(redW)])
    rowB = np.array([ry > 0 and (ry * upV) // ph != ((ry - 1) * upV) // ph for ry in range(redH)])
    return colB, rowB


def reach(bd):
    """fractions, over every (visit, mode) of every shape, of the piece borders where the reduced samples on both sides differ, and of
    the first reduced row / column that differ from the boundary sample the up-sampling reads at the same position"""
    orig, reco, visits, _, _ = case(bd)
    out = {}
    for v in visits:
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        x, y = int(v['x']), int(v['y'])
        if x == 0 or y == 0:
            continue
        top = reco[y - 1, x - 1:x + 2 * w].astype(np.int64)
        left = reco[y - 1:y + 2 * h, x - 1].astype(np.int64)
        redW, redH = min(w, 8), min(h, 8)
        upH, upV = w // redW, h // redH
        colB, rowB = unit_borders(w, h)
        r = out.setdefault((w, h), {'unit': [0, 0], 'bnd': [0, 0]})
        for mode in range(mip_num_modes(w, h)):
            red = mip_reduced(top, left, w, h, bd, mode)
            for rx in np.nonzero(colB)[0]:
                r['unit'][0] += int((red[:, rx] != red[:, rx - 1]).sum()); r['unit'][1] += redH
            for ry in np.nonzero(rowB)[0]:
                r['unit'][0] += int((red[ry] != red[ry - 1]).sum()); r['unit'][1] += redW
            if upV > 1:
                b = top[upH * np.arange(1, redW + 1)]
                r['bnd'][0] += int((red[0] != b).sum()); r['bnd'][1] += redW
            if upH > 1:
                b = left[upV * np.arange(1, redH + 1)]
                r['bnd'][0] += int((red[:, 0] != b).sum()); r['bnd'][1] += redH
    return out


@pytest.mark.parametrize('bd', BDS)
def test_cases_make_a_wrong_border_show(bd):
    r = reach(bd)
    assert set(r) == set(SHAPES)
    for shape, d in r.items():
        assert d['unit'][1] and d['unit'][0] >= 0.75 * d['unit'][1], (shape, d)
        assert d['bnd'][1] and d['bnd'][0] >= 0.75 * d['bnd'][1], (shape, d)


def every_mode_in_both_orientations(visits):
    n = {(1 << int(v['log2w']), 1 << int(v['log2h'])): mip_num_modes(1 << int(v['log2w']), 1 << int(v['log2h'])) for v in visits}
    return all(m == 11 for m in n.values())          # all modes 0..10 of the 16x16 family: 0..5 normal, 6..10 transposed


def assert_same(res, det, ora, odet):
    mip = slice(O.SLOT_MIP, O.SLOT_MIP + 11)
    bad = [i for i in range(len(res)) if det[i]['sad'][mip].tobytes() != odet[i]['sad'][mip].tobytes()
           or det[i]['satd'][mip].tobytes() != odet[i]['satd'][mip].tobytes()]
    assert not bad, bad[:5]
    assert det.tobytes() == odet.tobytes()
    assert res.tobytes() == ora.tobytes()


def mip_preds_match(pred, opred, w, h):
    for m in range(mip_num_modes(w, h)):
        if not np.array_equal(pred[O.SLOT_MIP + m], opred[O.SLOT_MIP + m]):
            return m
    return None


# ---- CPU tier: the kernel source on host threads ------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def emul():
    subprocess.check_call(['make', '-s', '-f', 'tests/host_emul/Makefile'], cwd=ROOT)
    return C.CDLL(os.path.join(ROOT, 'tests/host_emul/libemul_rmd.so'))


def run_emul(lib, orig, reco, bd, visits, pred=None):
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    visits = np.ascontiguousarray(visits, O.VISIT_DTYPE)
    res = np.zeros(len(visits), O.RESULT_DTYPE)
    det = np.zeros(len(visits), O.DETAIL_DTYPE)
    assert lib.emul_rmd_eval(p(orig), p(reco), orig.shape[1], bd, CTU, p(visits), len(visits), p(res), p(det),
                             p(pred) if pred is not None else None) == 0
    return res, det


@pytest.mark.parametrize('bd', BDS)
def test_emulated_sweep_sized_items(emul, bd):
    orig, reco, visits, ora, odet = case(bd)
    assert len(visits) > 96 and every_mode_in_both_orientations(visits)           # more than a walk-sized batch: per-bucket kernels
    res, det = run_emul(emul, orig, reco, bd, visits)
    assert_same(res, det, ora, odet)


@pytest.mark.parametrize('bd', BDS)
def test_emulated_walk_sized_batches(emul, bd):
    orig, reco, visits, ora, odet = case(bd)
    for lo in range(0, len(visits), 40):                                              # rmd_plan_small + rmd_eval_any_kernel
        sl = slice(lo, lo + 40)
        res, det = run_emul(emul, orig, reco, bd, visits[sl])
        assert_same(res, det, ora[sl], odet[sl])


@pytest.mark.parametrize('bd', BDS)
def test_emulated_prediction_output(emul, bd):
    orig, reco, visits, _, _ = case(bd)
    for k in range(1, len(visits), PER_SHAPE):       # one interior and (k - 1) one edge visit per shape
        for i in (k - 1, k + 1):
            v = visits[i:i + 1]
            w, h = 1 << int(v['log2w'][0]), 1 << int(v['log2h'][0])
            pred = np.zeros((O.NUM_SLOTS, h, w), np.int16)
            run_emul(emul, orig, reco, bd, v, pred)
            _, _, opreds = O.rmd_batch(orig, reco, bd, CTU, v, want_pred=True)
            assert mip_preds_match(pred, opreds[0], w, h) is None, ((w, h), int(v['x'][0]), int(v['y'][0]))


# ---- GPU tier: the library ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def engines():
    engs = {}
    yield lambda bd: engs.setdefault(bd, vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=CTU))
    for e in engs.values():
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize('bd', BDS)
def test_sweep_sized_and_walk_sized_calls(engines, bd):
    orig, reco, visits, ora, odet = case(bd)
    eng = engines(bd)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    # more than 4 096 visits: the per-bucket kernels of a sweep (packed and plain items); the same visits repeated
    reps = 4200 // len(visits) + 1
    res, det = eng.rmd_eval(np.tile(visits, reps), detail=True)
    assert_same(res, det, np.tile(ora, reps), np.tile(odet, reps))
    for lo in range(0, len(visits), 40):             # walk-sized: one launch for every bucket
        sl = slice(lo, lo + 40)
        res, det = eng.rmd_eval(visits[sl], detail=True)
        assert_same(res, det, ora[sl], odet[sl])


@pytest.mark.gpu
@pytest.mark.parametrize('bd', BDS)
def test_prediction_output(engines, bd):
    orig, reco, visits, _, _ = case(bd)
    eng = engines(bd)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    _, _, opreds = O.rmd_batch(orig, reco, bd, CTU, visits, want_pred=True)
    for v, op in zip(visits, opreds):
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        assert mip_preds_match(eng.rmd_pred_all(v), op, w, h) is None, ((w, h), int(v['x']), int(v['y']))
