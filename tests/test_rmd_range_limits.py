"""The rough-mode decision at the ends of its ranges: bit depths 8, 9 and 10, CTU sizes 32, 64 and 128, and reference lines that drive
MIP's inputs and every clip of the predictors to the sample range, against the oracle byte for byte.

Every visit sits on an atlas (as golden_util.build_atlas lays out recorded visits) whose cells hold its reference lines 0..3 and its
original block exactly, so the content of each line is chosen: 'split' (above at 0, left at max or the reverse: MIP inputs of +-max in
both orientations), 'segments' (each reduced-boundary segment 0 or max: MIP's reduced samples below 0 and above max before the clip),
'impulse' (one max sample in a zero line, or one zero in a max line: cubic-filter overshoot, [1 2 1] smoothing), 'check' (alternating
0 / max), 'corner' (only the top-left sample differs: PDPC's corner term).  Lines 1 and 3 differ from line 0, so a predictor that reads
the wrong line shows.  Originals are all 0, all max, a checkerboard, or the complement of the nearest reference sample.  The first visit
of every atlas row sits at x = 0, the first row at y = 0, the last cell of a row against the right edge and the last row against the
bottom edge; rows alternate between y on and off a multiple of 32, so at CTU sizes 32 and 64 some visits lose MRL to the CTU size alone.

Each case set also asserts that it reached what it is there for, from small numpy replicas of the kernels' arithmetic (MIP from the
kMip* tables of vvc_rom_tables.h, the cubic 4-tap filter, the PDPC of the pure horizontal / vertical modes, the 8x8 Hadamard DC).

GPU tier: vvcb_rmd_eval (with and without detail tables), vvcb_rmd_eval_brief, vvcb_rmd_pred_all, vvcb_tu_eval_pred with MRL slots and
vvcb_ctu_hads_islice, at every (bit depth, CTU size); the create refusals.  CPU tier: a subset of the same cases through the kernel
source on host threads (tests/host_emul); the device-only branches of vvcb_core.cuh (__dp2a_lo / __dp2a_hi, __vimin_s32_relu, __vmaxu2,
__sad) run only in the GPU tier."""
import ctypes as C
import functools
import os
import re
import subprocess

import numpy as np
import pytest

import vvc_intra_b200 as vb
from oracle import oracle_py as O
import golden_util as G
from test_kernel_emulation import brief_matches

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BDS = (8, 9, 10)
CTUS = (32, 64, 128)
SHAPES = [(lw, lh) for lw in range(2, 7) for lh in range(2, 7) if (lw == 6) == (lh == 6)]
FAMILIES = ('split', 'segments', 'impulse', 'check', 'corner')
ORIGINALS = ('zero', 'max', 'check', 'complement')
VARIANTS = {'split': 4, 'segments': 12, 'impulse': 2, 'check': 2, 'corner': 2}       # visits per (shape, family)
FULL = ('split', 'segments')        # families whose visits see their whole lines (available, MIP enabled) wherever the picture allows


# ---- content ------------------------------------------------------------------------------------------------------------------------
def line_pair(fam, var, w, h, bd, rng):
    """Reference line 0 of a family: (top, left), top[0] == left[0] the corner, top[1..2w] above and above-right, left[1..2h] left and
    below-left."""
    mx = (1 << bd) - 1
    top, left = np.zeros(2 * w + 1, np.int64), np.zeros(2 * h + 1, np.int64)
    if fam == 'split':                               # normal orientation: in[i >= bsz] = +-max, transposed: in[i < bsz] = -+max
        top[:], left[:] = (0, mx) if var == 0 else (mx, 0)
        left[0] = top[0] = int(rng.integers(0, 2)) * mx
    elif fam == 'segments':                          # the reduced-boundary segments (w / bsz, h / bsz samples) independently 0 or max
        bsz = 4 if (w > 4 or h > 4) else 2
        top[1:w + 1] = np.repeat(rng.integers(0, 2, bsz), w // bsz) * mx
        left[1:h + 1] = np.repeat(rng.integers(0, 2, bsz), h // bsz) * mx
        top[w + 1:] = np.repeat(rng.integers(0, 2, w // 4), 4) * mx
        left[h + 1:] = np.repeat(rng.integers(0, 2, h // 4), 4) * mx
        left[0] = top[0] = int(rng.integers(0, 2)) * mx
    elif fam == 'impulse':                           # var 0: one max sample in a zero line, var 1: one zero in a max line
        base = 0 if var == 0 else mx
        top[:], left[:] = base, base
        k = int(rng.integers(0, 2 * (w + h) + 1))
        if k <= 2 * w:
            top[k] = mx - base
        else:
            left[k - 2 * w] = mx - base
        left[0] = top[0]
    elif fam == 'check':
        top[:] = ((np.arange(2 * w + 1) + var) & 1) * mx
        left[:] = ((np.arange(2 * h + 1) + var) & 1) * mx
        left[0] = top[0]
    else:                                            # 'corner': everything a, the top-left sample max - a
        a = mx if var == 0 else 0
        top[:], left[:] = a, a
        top[0] = left[0] = mx - a
    return top, left


def mrl_lines(top, left, bd, rng):
    """Lines 1, 2, 3 from line 0: line 1 the complement, line 2 (read by nothing) and line 3 line 0 rotated, so that each differs from
    line 0 and from each other wherever line 0 is not flat"""
    mx = (1 << bd) - 1
    out = {0: (top, left)}
    for m in (1, 2, 3):
        if m == 1:
            t, l = mx - top, mx - left
        else:
            s = int(rng.integers(1, 4))
            t, l = np.roll(top, s), np.roll(left, s)
            if not (t != top).any():                 # a flat line: line 3 its complement at the far end
                t, l = t.copy(), l.copy()
                t[len(t) // 2:] = mx - t[len(t) // 2:]
                l[len(l) // 2:] = mx - l[len(l) // 2:]
        t = np.concatenate([t, t[-1:].repeat(m)])
        l = np.concatenate([l, l[-1:].repeat(m)])
        l[0] = t[0]
        out[m] = (t, l)
    return out


def original(kind, top, left, w, h, bd):
    mx = (1 << bd) - 1
    y, x = np.mgrid[0:h, 0:w]
    if kind == 'zero':
        return np.zeros((h, w), np.int64)
    if kind == 'max':
        return np.full((h, w), mx, np.int64)
    if kind == 'check':
        return ((x + y) & 1) * mx
    return mx - np.where(x >= y, top[1 + x], left[1 + y])        # complement of the nearest reference sample


def random_visit_fields(v, rng, w, h):
    """availability (all / none / ragged), NO_MRL / NO_MIP flags, random MPM list, rates and lambda"""
    mode = rng.choice(4, p=[0.6, 0.1, 0.15, 0.15])
    if mode == 0:
        v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = 1, w // 4, w // 4, h // 4, h // 4
    elif mode >= 2:
        v['avail_al'] = rng.integers(0, 2)
        v['n_above'], v['n_above_right'] = rng.integers(0, w // 4 + 1, 2)
        v['n_left'], v['n_below_left'] = rng.integers(0, h // 4 + 1, 2)
    v['flags'] = rng.choice(4, p=[0.7, 0.1, 0.1, 0.1])
    L, A = rng.integers(0, 67, 2)
    mpm, nc = O.intra_mpms(int(L), int(A))
    v['mpm'], v['num_mpm_cand'] = mpm, nc
    v['rates'] = rng.integers(100, 200000, 11)
    v['sqrt_lambda'] = float(rng.uniform(1e-4, 3e-3))


def structured_case(bd, ctu, seed, atlas_w=1024, families=FAMILIES):
    """-> (orig, reco, visits, tags): one visit per (shape, family, variant) with its lines and original written into an atlas cell.
    tags[i] = (family, original kind)."""
    rng = np.random.default_rng(seed)
    items = []
    for lw, lh in SHAPES:
        w, h = 1 << lw, 1 << lh
        for fam in families:
            for var in range(VARIANTS[fam]):
                top, left = line_pair(fam, var % 2 if fam != 'segments' else var, w, h, bd, rng)
                lines = mrl_lines(top, left, bd, rng)
                kind = ORIGINALS[(len(items) + var) % len(ORIGINALS)]
                items.append(dict(lw=lw, lh=lh, lines=lines, org=original(kind, top, left, w, h, bd), tag=(fam, kind), full=fam in FULL))
    order = rng.permutation(len(items))
    items = [items[i] for i in order]
    # rows of cells: a CU and its lines 0..3 (above, above-right, left, below-left); the first CU of a row at x = 0, the first row at
    # y = 0, the last CU of a row flush with the right edge, the last row flush with the bottom edge.  The CUs of a row share y: 16 modulo
    # 32 on even rows (no CTU row), 0, 32, 64, 96 modulo 128 in turn on odd rows (rows of CTUs of 32, 64 and 128)
    rows, cur, x = [], [], 0
    for it in items:
        cw = 2 * (1 << it['lw']) + 8
        if x + cw > atlas_w:
            rows.append(cur)
            cur, x = [], 0
        cur.append(it)
        x += cw
    rows.append(cur)
    y, bottom = 0, 0
    for r, row in enumerate(rows):
        if r:
            target = 16 if r % 2 == 0 else 32 * ((r // 2) % 4)
            y = bottom + 4 + (target - bottom - 4) % (32 if r % 2 == 0 else 128)
        x = 0
        for k, it in enumerate(row):
            it['x'], it['y'] = (0 if k == 0 else x + 4), y
            x = it['x'] + 2 * (1 << it['lw'])
        row[-1]['x'] = atlas_w - (1 << row[-1]['lw'])
        bottom = y + max(2 * (1 << it['lh']) for it in row)
    H = max(it['y'] + (1 << it['lh']) for it in rows[-1])
    for it in rows[-1]:
        it['y'] = H - (1 << it['lh'])
    W = atlas_w
    orig = np.zeros((H, W), np.int16)
    reco = np.full((H, W), (1 << bd) >> 1, np.int16)
    visits = np.zeros(len(items), O.VISIT_DTYPE)
    tags = []
    for i, it in enumerate(items):
        w, h, x0, y0 = 1 << it['lw'], 1 << it['lh'], it['x'], it['y']
        for m in (3, 2, 1, 0):
            t, l = it['lines'][m]
            xs, ys = x0 - 1 - m + np.arange(len(t)), np.full(len(t), y0 - 1 - m)
            ok = (xs >= 0) & (xs < W) & (ys >= 0)
            reco[ys[ok], xs[ok]] = t[ok]
            xs, ys = np.full(len(l), x0 - 1 - m), y0 - 1 - m + np.arange(len(l))
            ok = (xs >= 0) & (ys >= 0) & (ys < H)
            reco[ys[ok], xs[ok]] = l[ok]
        orig[y0:y0 + h, x0:x0 + w] = it['org']
        v = visits[i]
        v['x'], v['y'], v['log2w'], v['log2h'] = x0, y0, it['lw'], it['lh']
        random_visit_fields(v, rng, w, h)
        if it['full']:
            v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = 1, w // 4, w // 4, h // 4, h // 4
            v['flags'] &= 1
        if y0 < 4:
            v['avail_al'], v['n_above'], v['n_above_right'] = 0, 0, 0
        if x0 < 4:
            v['avail_al'], v['n_left'], v['n_below_left'] = 0, 0, 0
        v['n_above_right'] = min(int(v['n_above_right']), (W - x0 - w) // 4)
        v['n_below_left'] = min(int(v['n_below_left']), (H - y0 - h) // 4)
        tags.append(it['tag'])
    return orig, reco, visits, tags


@functools.lru_cache(maxsize=None)
def case(bd, ctu):
    """the structured case of (bd, ctu) and the oracle's results, details and prediction samples of every slot"""
    orig, reco, visits, tags = structured_case(bd, ctu, 1000 * bd + ctu)
    res, det, preds = O.rmd_batch(orig, reco, bd, ctu, visits, want_pred=True)
    return orig, reco, visits, tags, res, det, preds


def random_ctu_case(bd, ctu, seed, n_per_shape=6):
    """golden_util.random_case with a third of the visits moved onto a multiple of the CTU size that is not a multiple of 128 (for
    CTU 128: onto a multiple of 128)"""
    rng = np.random.default_rng(seed)
    orig, reco, arr = G.random_case(rng, bd, n_per_shape, plane=(512, 512))
    on_row = rng.random(len(arr)) < 0.33
    step = ctu if ctu < 128 else 128
    ys = step * (2 * rng.integers(0, 512 // (2 * step), len(arr)) + (1 if ctu < 128 else 0))
    fits = ys + (1 << arr['log2h'].astype(np.int64)) * 2 <= 512
    sel = on_row & fits & (ys >= 4)
    arr['y'][sel] = ys[sel]
    return orig, reco, arr


# ---- replicas of the kernels' arithmetic (reach) ----------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def rom_tables():
    txt = open(os.path.join(ROOT, 'vvc_intra_b200/csrc/vvc_rom_tables.h')).read()
    return {m.group(1): np.array([int(v) for v in m.group(2).split(',') if v.strip()], np.int64)
            for m in re.finditer(r'static const u?int8_t (k(?:Mip|Intra)\w+)\[\d+\] = \{([^}]*)\}', txt)}


def mip_family(w, h):
    return 0 if w == h == 4 else (1 if w <= 8 and h <= 8 else 2)


def mip_num_modes(w, h):
    if w > 4 * h or h > 4 * w:
        return 0
    return 35 if w == h == 4 else (19 if w <= 8 and h <= 8 else 11)


def mip_reach(top, left, w, h, bd, r):
    """orc_pred_mip's / mip_row_sample's arithmetic up to the clip, for every mode of the block: records the input vectors of both
    orientations and the reduced samples before the clip, per (family, transposed)"""
    T = rom_tables()
    fam = mip_family(w, h)
    n = mip_num_modes(w, h)
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
    mx = (1 << bd) - 1
    for t in (0, 1):
        inp = np.concatenate([bL, bT] if t else [bT, bL])
        first = int(inp[0])
        inp[1:] -= first
        inp[0] = first - (1 << (bd - 1)) if small else 0
        key = (fam, t)
        r['in_abs'][key] = max(r['in_abs'].get(key, 0), int(np.abs(inp[1:]).max()))
        if small:
            r['in0'].setdefault(fam, set()).add(int(inp[0]))
        lho, lvo = (w == 4 and h >= 16), (h == 4 and w >= 16)
        iw, ih = (redH, redW) if t else (redW, redH)
        if t:
            lho, lvo = lvo, lho
        yy, xx = np.mgrid[0:ih, 0:iw]
        rows = ((2 * yy if lvo else yy) * (iw if small else 8) + (2 * xx if lho else xx)).ravel()
        for widx in (range(1, n // 2 + 1) if t else range(n // 2 + 1)):
            M = mats[widx * rows_ * cols:(widx + 1) * rows_ * cols].reshape(rows_, cols)[rows]
            acc = M @ (inp if small else inp[1:])
            off = (1 << (int(shifts[widx]) - 1)) - int(offs[widx]) * int(inp.sum())
            v = ((acc + off) >> int(shifts[widx])) + first
            k = (fam, t, widx)
            lo, hi = r['mip'].get(k, (0, mx))
            r['mip'][k] = (min(lo, int(v.min())), max(hi, int(v.max())))


@functools.lru_cache(maxsize=None)
def ipa(w, h, mode, mrl):
    p = O.ipa_init(w, h, mode, mrl)
    return p.is_ver, p.ref_filter, p.interp, p.pdpc, p.angle, p.inv_angle


def angular_reach(top, left, w, h, bd, mode, mrl, r):
    """pred_angular_unit's 4-tap cubic filter before its clip (slots on an unfiltered line with a fractional slope and the cubic
    filter), and the PDPC of the pure horizontal / vertical modes before its clip"""
    is_ver, ref_filter, interp, pdpc, angle, inv_angle = ipa(w, h, mode, mrl)
    if ref_filter or (angle != 0 and (interp or not (abs(angle) & 31))):
        return
    main, side = (top, left) if is_ver else (left, top)
    mw, mh = (w, h) if is_ver else (h, w)
    main, side = main.astype(np.int64), side.astype(np.int64)
    if angle == 0:
        if pdpc:
            scale = ((mw.bit_length() - 1) + (mh.bit_length() - 1) - 2) >> 2
            c = np.arange(min(3 << scale, mw))
            wL = 32 >> ((2 * c) >> scale)
            v = main[1 + c][None, :] + ((wL[None, :] * (side[1:1 + mh, None] - main[0]) + 32) >> 6)
            r['pdpc'] = (min(r['pdpc'][0], int(v.min())), max(r['pdpc'][1], int(v.max())))
        return
    OFF = 2 * 64 + 8
    buf = np.zeros(OFF + 2 * 64 + 16, np.int64)
    if angle < 0:
        buf[OFF:OFF + mw + 2 + mrl] = main[:mw + 2 + mrl]
        i = np.arange(-mh, 0)
        buf[OFF + i] = side[np.minimum((-i * inv_angle + 256) >> 9, mh)]
    else:
        ml = 2 * mw
        ext = (mrl << max(0, (mw.bit_length() - mh.bit_length()))) + 2
        buf[OFF:OFF + ml + mrl + 1] = main[:ml + mrl + 1]
        buf[OFF + ml + mrl + 1:OFF + ml + mrl + 1 + ext] = main[ml + mrl]
    rr = np.arange(mh)
    pos = angle * (rr + 1 + mrl)
    d_int, d_frac = pos >> 5, pos & 31
    f = rom_tables()['kIntraCubicFilter'].reshape(32, 4)[d_frac]
    idx = OFF + mrl + d_int[:, None] + np.arange(mw)[None, :]
    v = (sum(f[:, k, None] * buf[idx + k] for k in range(4)) + 32) >> 6
    r['cubic'] = (min(r['cubic'][0], int(v.min())), max(r['cubic'][1], int(v.max())))


def reach(orig, reco, visits, tags, det, preds, bd, ctu):
    """the replicas over every visit, per content family"""
    mx = (1 << bd) - 1
    out = dict(mrl_off_by_ctu=0)
    for i, v in enumerate(visits):
        r = out.setdefault(tags[i][0], dict(in_abs={}, in0={}, mip={}, cubic=(0, mx), pdpc=(0, mx), had_dc=0))
        w, h, x, y = 1 << int(v['log2w']), 1 << int(v['log2h']), int(v['x']), int(v['y'])
        args = (int(v['avail_al']), int(v['n_above']), int(v['n_above_right']), int(v['n_left']), int(v['n_below_left']))
        lines = {m: O.ref_fill(reco, x, y, w, h, m, bd, *args) for m in (0, 1, 3)}
        mrl_ok = not (int(v['flags']) & 1) and y % ctu != 0
        if not (int(v['flags']) & 1) and y % ctu == 0 and y % 128 != 0:
            out['mrl_off_by_ctu'] += 1
        if not (int(v['flags']) & 2) and mip_num_modes(w, h):
            mip_reach(*lines[0], w, h, bd, r)
        for mode in range(2, 67):
            angular_reach(*lines[0], w, h, bd, mode, 0, r)
        if mrl_ok:
            for m in (1, 3):
                for mode in set(int(k) for k in v['mpm'][1:]) - {0, 1}:
                    angular_reach(*lines[m], w, h, bd, mode, m, r)
        if w % 8 == 0 and h % 8 == 0:
            ev = np.flatnonzero(det[i]['sad'] != O.SAT_NONE)
            res = orig[y:y + h, x:x + w].astype(np.int64)[None] - preds[i][ev].astype(np.int64)
            dc = np.abs(res.reshape(len(ev), h // 8, 8, w // 8, 8).sum((2, 4))).max()
            r['had_dc'] = max(r['had_dc'], int(dc))
    return out


def reach_failures(out, bd, ctu):
    """names of the edges the case set did not reach, each from the content family that is there to reach it"""
    mx = (1 << bd) - 1
    empty = dict(in_abs={}, in0={}, mip={}, cubic=(0, mx), pdpc=(0, mx), had_dc=0)
    fam_of = lambda f: out.get(f, empty)
    missed = []
    for fam in (0, 1, 2):
        for t in (0, 1):
            if fam_of('split')['in_abs'].get((fam, t)) != mx:
                missed.append('split: MIP |in[i >= 1]| = max, family %d, transposed %d' % (fam, t))
            modes = {k: v for k, v in fam_of('segments')['mip'].items() if k[:2] == (fam, t)}
            if not modes or not all(lo < 0 and hi > mx for lo, hi in modes.values()):
                missed.append('segments: MIP reduced sample below 0 and above max before the clip, family %d, transposed %d, every mode' % (fam, t))
    for fam in (0, 1):
        if not {-(1 << (bd - 1)), (1 << (bd - 1)) - 1} <= fam_of('split')['in0'].get(fam, set()):
            missed.append('split: MIP in[0] at both ends, family %d' % fam)
    for f in ('impulse', 'check'):
        if not (fam_of(f)['cubic'][0] < 0 and fam_of(f)['cubic'][1] > mx):
            missed.append('%s: cubic filter below 0 and above max' % f)
    if not (fam_of('corner')['pdpc'][0] < 0 and fam_of('corner')['pdpc'][1] > mx):
        missed.append('corner: PDPC of the pure horizontal / vertical modes below 0 and above max')
    if fam_of('split')['had_dc'] != 64 * mx:
        missed.append('split: 8x8 Hadamard |DC| = 64 max')
    if ctu < 128 and not out['mrl_off_by_ctu']:
        missed.append('MRL turned off by the CTU size alone')
    return missed


def assert_reach(r, bd, ctu):
    missed = reach_failures(r, bd, ctu)
    assert not missed, missed


@functools.lru_cache(maxsize=None)
def case_reach(bd, ctu):
    orig, reco, visits, tags, res, det, preds = case(bd, ctu)
    return reach(orig, reco, visits, tags, det, preds, bd, ctu)


# ---- comparisons ---------------------------------------------------------------------------------------------------------------------
def assert_same(res, det, ora, odet, visits, tags=None):
    bad = [i for i in range(len(visits)) if res[i].tobytes() != ora[i].tobytes() or det[i].tobytes() != odet[i].tobytes()]
    assert not bad, (len(bad), visits[bad[0]], tags[bad[0]] if tags else None,
                     [s for s in range(O.NUM_SLOTS) if det[bad[0]]['satd'][s] != odet[bad[0]]['satd'][s] or det[bad[0]]['sad'][s] != odet[bad[0]]['sad'][s]][:10])


def pred_subset(visits, tags):
    """one visit per (shape, family)"""
    seen, out = set(), []
    for i, (v, t) in enumerate(zip(visits, tags)):
        k = (int(v['log2w']), int(v['log2h']), t[0])
        if k not in seen:
            seen.add(k)
            out.append(i)
    return out


def tu_pred_jobs(rng, bd, ctu, orig, visits, preds, per_visit=3):
    """Like golden_util.pred_tu_case for a given CTU size: per visit a regular slot, an MRL slot wherever the CTU size allows one and a
    MIP slot wherever the visit evaluates MIP, each one dependent-quantisation TU job.  Returns (src, jobs, n_samples, rates, items)."""
    n_rates = 3
    rates = np.zeros(n_rates, vb.DQ_RATES_DTYPE)
    for name in rates.dtype.names:
        rates[name] = rng.integers(300, 140000, rates[name].shape)
    src, jobs, items, off = [], [], [], 0
    for vi, v in enumerate(visits):
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        mrl_ok = not (int(v['flags']) & 1) and (int(v['y']) & (ctu - 1)) != 0
        n_mip = 0 if int(v['flags']) & 2 else mip_num_modes(w, h)
        cand = [int(rng.integers(0, 67))]
        if mrl_ok:
            cand.append(int(rng.choice([O.SLOT_MRL1, O.SLOT_MRL3])) + int(rng.integers(0, 5)))
        if n_mip:
            cand.append(O.SLOT_MIP + int(rng.integers(0, n_mip)))
        for slot in cand[:per_visit]:
            mts = int(rng.choice([0, 0, 2, 5])) if max(w, h) <= 32 else 0
            qp = int(rng.integers(16, 48)) + 6 * (bd - 8)
            j = np.zeros(1, vb.TU_JOB_DTYPE)[0]
            j['x'], j['y'], j['log2w'], j['log2h'], j['mts_idx'] = v['x'], v['y'], v['log2w'], v['log2h'], mts
            j['flags'] = vb.TU_QUANT | vb.TU_DEPQUANT
            j['qp_per'], j['qp_rem'], j['offset'] = qp // 6, qp % 6, off
            lam = float(0.57 * 2.0 ** ((qp - 6 * (bd - 8) - 12) / 3.0))
            j['rate_idx'], j['cbf_delta_bits'], j['lambda'] = len(jobs) % n_rates, int(rng.integers(-30000, 30000)), lam
            p = preds[vi][slot]
            o = orig[int(v['y']):int(v['y']) + h, int(v['x']):int(v['x']) + w]
            items.append(dict(pred=p, org=o, resi=(o.astype(np.int32) - p).astype(np.int16), mts=mts, qp=qp, lam=lam, cbf=int(j['cbf_delta_bits']),
                              lfnst=0, intra=0, off=off, rate=rates[len(jobs) % n_rates]))
            s = np.zeros(1, vb.TU_SRC_DTYPE)[0]
            s['visit'], s['slot'] = vi, slot
            src.append(s)
            jobs.append(j)
            off += w * h
    return np.array(src, vb.TU_SRC_DTYPE), np.array(jobs, vb.TU_JOB_DTYPE), off, rates, items


def hads_pictures(bd):
    """full-scale pictures whose sizes are not multiples of the CTU: 0 / max checkerboard blocks, 0 / max random samples, noise"""
    mx = (1 << bd) - 1
    rng = np.random.default_rng(bd)
    out = []
    for H, W in ((136, 200), (240, 416)):
        y, x = np.mgrid[0:H, 0:W]
        out.append(((x + y) & 1) * mx)
        out.append(rng.integers(0, 2, (H, W)) * mx)
        out.append(rng.integers(0, mx + 1, (H, W)))
    return [p.astype(np.int16) for p in out]


# ---- GPU tier ----------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def engines():
    cache = {}

    def get(bd, ctu):
        if (bd, ctu) not in cache:
            cache[(bd, ctu)] = vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=ctu)
        return cache[(bd, ctu)]
    yield get
    for e in cache.values():
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize('ctu', CTUS)
@pytest.mark.parametrize('bd', BDS)
def test_rmd_at_the_range_limits(bd, ctu, engines):
    """the structured case: results and detail tables, the results without detail (min(2 SAD, SATD) hand-off), the brief records"""
    eng = engines(bd, ctu)
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    res, det = eng.rmd_eval(visits, detail=True)
    assert_same(res, det, ora, odet, visits, tags)
    assert eng.rmd_eval(visits).tobytes() == ora.tobytes()
    assert brief_matches(eng.rmd_eval_brief(visits), ora)
    # walk-sized batches (one plan kernel, one launch per item flavour) of the same visits
    for k in range(0, len(visits), 61):
        assert eng.rmd_eval(visits[k:k + 61]).tobytes() == ora[k:k + 61].tobytes()
    assert_reach(case_reach(bd, ctu), bd, ctu)


@pytest.mark.gpu
@pytest.mark.parametrize('ctu', CTUS)
@pytest.mark.parametrize('bd', BDS)
def test_prediction_samples_at_the_range_limits(bd, ctu, engines):
    """vvcb_rmd_pred_all: the samples of every slot of one visit per (shape, family) against the oracle's; the slots the visit does not
    evaluate keep what the caller's buffer held"""
    eng = engines(bd, ctu)
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    sel = pred_subset(visits, tags)
    assert len(sel) == len(SHAPES) * len(FAMILIES)
    skipped = 0
    for i in sel:
        w, h = 1 << int(visits[i]['log2w']), 1 << int(visits[i]['log2h'])
        got = np.full((O.NUM_SLOTS, h, w), -1, np.int16)
        eng._ck(eng._lib.vvcb_rmd_pred_all(eng._ctx, C.c_void_p(visits[i:i + 1].ctypes.data), C.c_void_p(got.ctypes.data)))
        ev = odet[i]['sad'] != O.SAT_NONE
        bad = [s for s in range(O.NUM_SLOTS) if not np.array_equal(got[s], preds[i][s] if ev[s] else np.full((h, w), -1))]
        assert not bad, (tags[i], visits[i], bad[:10])
        skipped += int((~ev[:O.SLOT_MIP]).any())
    assert skipped > 0


@pytest.mark.gpu
@pytest.mark.parametrize('ctu', (32, 64))
@pytest.mark.parametrize('bd', BDS)
def test_random_visits_at_small_ctu_sizes(bd, ctu, engines):
    """noise content with visits on CTU rows that are not rows of a 128 CTU; the small shapes alone as packed items, a third of them on
    CTU rows, in walk-sized and in larger batches"""
    eng = engines(bd, ctu)
    orig, reco, arr = random_ctu_case(bd, ctu, 10 * bd + ctu)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    ora, odet = O.rmd_batch(orig, reco, bd, ctu, arr)
    res, det = eng.rmd_eval(arr, detail=True)
    assert_same(res, det, ora, odet, arr)
    assert eng.rmd_eval(arr).tobytes() == ora.tobytes()
    assert brief_matches(eng.rmd_eval_brief(arr), ora)
    small = np.isin(arr['log2w'] * 8 + arr['log2h'], [lw * 8 + lh for lw, lh in [(2, 2), (3, 2), (2, 3), (3, 3), (4, 2), (2, 4), (4, 3), (3, 4)]])
    sm = arr[small]
    on_row = (sm['y'] % ctu == 0) & (sm['flags'] & 1 == 0)
    assert on_row.any() and (~on_row).any()
    for part in (sm[:90], sm):
        ps = O.rmd_batch(orig, reco, bd, ctu, part)[0]
        assert eng.rmd_eval(part).tobytes() == ps.tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize('ctu', (32, 64))
@pytest.mark.parametrize('bd', BDS)
def test_tu_eval_pred_at_small_ctu_sizes(bd, ctu, engines):
    """vvcb_tu_eval_pred with regular, MRL and MIP slots of the structured visits; an MRL slot of a visit on a CTU row is refused"""
    eng = engines(bd, ctu)
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    rng = np.random.default_rng(bd * 100 + ctu)
    src, jobs, n_samples, rates, items = tu_pred_jobs(rng, bd, ctu, orig, visits, preds)
    assert (src['slot'] >= O.SLOT_MRL1).any() and ((src['slot'] >= O.SLOT_MRL1) & (src['slot'] < O.SLOT_MIP)).any()
    out = eng.tu_eval_pred(visits, src, jobs, n_samples, want_coeff=True, want_level=True, want_reco=True, want_pred=True, rates=rates)
    exp = G.oracle_dq_chain(items, bd)
    for i, it in enumerate(items):
        sl = slice(it['off'], it['off'] + it['pred'].size)
        assert np.array_equal(out['pred'][sl].reshape(it['pred'].shape), it['pred']), (i, tags[int(src[i]['visit'])], int(src[i]['slot']))
    for k in ('coeff', 'level', 'reco'):
        assert np.array_equal(out[k], exp[k]), k
    assert out['results'].tobytes() == exp['results'].tobytes()
    row = [i for i, v in enumerate(visits) if int(v['y']) % ctu == 0 and int(v['y']) % 128 != 0 and not int(v['flags']) & 1]
    assert row
    bad = src[:1].copy()
    bad['visit'], bad['slot'] = row[0], O.SLOT_MRL1
    badj = jobs[:1].copy()
    for k in ('x', 'y', 'log2w', 'log2h'):
        badj[k] = visits[row[0]][k]
    badj['mts_idx'] = 0
    with pytest.raises(vb.EngineError, match='malformed'):
        eng.tu_eval_pred(visits, bad, badj, 1 << (int(badj['log2w'][0]) + int(badj['log2h'][0])), rates=rates)
    with pytest.raises(vb.EngineError, match='not evaluated'):
        eng.rmd_pred(visits[row[0]], O.SLOT_MRL1)


@pytest.mark.gpu
@pytest.mark.parametrize('ctu', CTUS)
@pytest.mark.parametrize('bd', BDS)
def test_ctu_hads_at_every_ctu_size(bd, ctu, engines):
    eng = engines(bd, ctu)
    for pic in hads_pictures(bd):
        eng.frame_begin(pic)
        assert eng.ctu_hads_islice(pic.shape[1], pic.shape[0]).tolist() == O.ctu_hads_islice(pic, ctu=ctu).tolist(), pic.shape


# ---- refusals (the arguments are checked before any device is looked for: no GPU needed) ---------------------------------------------
REFUSED = [(7, 128), (11, 128), (12, 128), (10, 16), (10, 256), (8, 512), (9, 48), (9, 0)]


@pytest.mark.parametrize('bd,ctu', REFUSED)
def test_create_refuses_bit_depths_and_ctu_sizes_outside_the_supported_range(bd, ctu):
    """bit depths outside 8..10 and CTU sizes other than 32, 64 and 128 (H.266: CtbSizeY = 1 << (sps_log2_ctu_size_minus5 + 5), the
    syntax element at most 2)"""
    vb.engine.load_library()
    with pytest.raises(vb.EngineError, match='bad argument'):
        vb.IntraCostEngine(device=0, bit_depth=bd, ctu_size=ctu)


@pytest.mark.parametrize('bd,ctu', REFUSED + [(8, 32), (9, 64), (10, 128)])
def test_cpu_stand_in_refuses_what_the_library_refuses(bd, ctu):
    subprocess.check_call(['make', '-s', '-f', 'tests/fake_engine/Makefile'], cwd=ROOT)
    lib = C.CDLL(os.path.join(ROOT, 'tests/fake_engine/libvvc_intra_b200.so'))
    ctx = C.c_void_p()
    rc = lib.vvcb_create(C.byref(ctx), 0, bd, ctu)
    if (bd, ctu) in REFUSED:
        assert rc != 0 and not ctx.value
    else:
        assert rc == 0 and ctx.value
        lib.vvcb_destroy(ctx)


# ---- CPU tier: the kernel source on host threads ------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def emul():
    subprocess.check_call(['make', '-s', '-f', 'tests/host_emul/Makefile'], cwd=ROOT)
    return C.CDLL(os.path.join(ROOT, 'tests/host_emul/libemul_rmd.so'))


def run_emul(lib, orig, reco, bd, ctu, visits, detail=True):
    """test_kernel_emulation.run_emul with the CTU size passed through"""
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    orig, reco = np.ascontiguousarray(orig, np.int16), np.ascontiguousarray(reco, np.int16)
    visits = np.ascontiguousarray(visits, O.VISIT_DTYPE)
    res = np.zeros(len(visits), O.RESULT_DTYPE)
    det = np.zeros(len(visits), O.DETAIL_DTYPE)
    assert lib.emul_rmd_eval(p(orig), p(reco), orig.shape[1], bd, ctu, p(visits), len(visits), p(res), p(det) if detail else None, None) == 0
    return res, det


def emul_subset(visits, tags, per_shape):
    """per_shape visits of every shape, of different families, the families taken in turn over the shapes"""
    first = {}
    for i, (v, t) in enumerate(zip(visits, tags)):
        first.setdefault((int(v['log2w']), int(v['log2h']), t[0]), i)
    return np.array(sorted(first[(lw, lh, FAMILIES[(k + j) % len(FAMILIES)])] for k, (lw, lh) in enumerate(SHAPES) for j in range(per_shape)))


EMUL_CASES = [(bd, ctu) for bd in BDS for ctu in CTUS]


@pytest.mark.parametrize('bd,ctu', EMUL_CASES)
def test_emulated_rmd_at_the_range_limits(emul, bd, ctu):
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    sel = emul_subset(visits, tags, 2)
    sub = visits[sel]
    res, det = run_emul(emul, orig, reco, bd, ctu, sub)
    assert_same(res, det, ora[sel], odet[sel], sub, [tags[i] for i in sel])
    res2, _ = run_emul(emul, orig, reco, bd, ctu, sub, detail=False)
    assert res2.tobytes() == ora[sel].tobytes()
    brief = np.zeros(len(sub), vb.BRIEF_DTYPE)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert emul.emul_rmd_brief(p(sub), len(sub), ctu, p(np.ascontiguousarray(odet[sel])), p(brief)) == 0
    assert brief_matches(brief, ora[sel])


@pytest.mark.parametrize('bd,ctu', EMUL_CASES)
def test_emulated_tu_prediction_at_every_ctu_size(emul, bd, ctu):
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    sel = emul_subset(visits, tags, 1)
    rng = np.random.default_rng(bd * 100 + ctu + 1)
    src, jobs, n_samples, rates, items = tu_pred_jobs(rng, bd, ctu, orig, visits[sel], [preds[i] for i in sel])
    assert ((src['slot'] >= O.SLOT_MRL1) & (src['slot'] < O.SLOT_MIP)).any() and (src['slot'] >= O.SLOT_MIP).any()
    pred, resi = np.zeros(n_samples, np.int16), np.zeros(n_samples, np.int16)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    sub = np.ascontiguousarray(visits[sel])
    emul.emul_tu_pred(p(orig), p(reco), orig.shape[1], bd, ctu, p(sub), p(src), p(jobs), len(jobs), p(pred), p(resi))
    for s, it in zip(src, items):
        sl = slice(it['off'], it['off'] + it['pred'].size)
        assert np.array_equal(pred[sl].reshape(it['pred'].shape), it['pred']), (it['pred'].shape, int(s['slot']))
        assert np.array_equal(resi[sl].reshape(it['pred'].shape), it['resi']), (it['pred'].shape, int(s['slot']))


@pytest.mark.parametrize('ctu', CTUS)
def test_emulated_ctu_hads_at_every_ctu_size(emul, ctu):
    for bd in BDS:
        for pic in hads_pictures(bd):
            H, W = pic.shape
            out = np.zeros(-(-W // ctu) * -(-H // ctu), np.int32)
            emul.emul_ctu_hads(pic.ctypes.data_as(C.c_void_p), W, W, H, ctu, out.ctypes.data_as(C.c_void_p))
            assert out.tolist() == O.ctu_hads_islice(pic, ctu=ctu).tolist(), (bd, pic.shape)


# ---- the cases reach what they are there for ---------------------------------------------------------------------------------------
@pytest.mark.parametrize('ctu', CTUS)
@pytest.mark.parametrize('bd', BDS)
def test_cases_reach_the_range_limits(bd, ctu):
    assert_reach(case_reach(bd, ctu), bd, ctu)
    orig, reco, visits, tags, ora, odet, preds = case(bd, ctu)
    assert (visits['x'] == 0).any() and (visits['y'] == 0).any()
    assert (visits['x'] + (1 << visits['log2w'].astype(np.int64)) == orig.shape[1]).any()
    assert (visits['y'] + (1 << visits['log2h'].astype(np.int64)) == orig.shape[0]).any()
    full = (visits['avail_al'] == 1) & (visits['n_above'] > 0) & (visits['n_left'] > 0)
    assert full.sum() > len(visits) // 2 and (visits['flags'] & 1).any() and (visits['flags'] & 2).any()


def test_each_edge_needs_its_family():
    """without its content family, each family's edges above go unreached"""
    bd, ctu = 10, 64
    for drop in FAMILIES:
        orig, reco, visits, tags = structured_case(bd, ctu, 1000 * bd + ctu, families=tuple(f for f in FAMILIES if f != drop))
        res, det, preds = O.rmd_batch(orig, reco, bd, ctu, visits, want_pred=True)
        missed = reach_failures(reach(orig, reco, visits, tags, det, preds, bd, ctu), bd, ctu)
        assert any(m.startswith(drop + ':') for m in missed), (drop, missed)
