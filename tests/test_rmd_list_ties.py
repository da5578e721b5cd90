"""The candidate lists of the list kernel (vvc_intra_b200/csrc/vvcb_rmd.cuh, rmd_lists_kernel, run on host threads through
tests/host_emul/cuda_emul.h) against the oracle where many candidates tie.  updateCandList keeps equal costs in arrival order, so
a list built in any other order than the reference's pushes (by rank, in parallel) breaks ties the wrong way.  Random pictures rarely produce ties:
flat and periodic pictures make many modes' SAD and SATD equal, equal rates make their bits equal, and a zero lambda makes every
RD cost its distance.  Every CU shape, on and off CTU rows, with and without MIP, 8 and 10 bits."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle_py as O
from test_kernel_emulation import brief_matches, emul, run_emul  # noqa: F401  (emul is a fixture)

SHAPES = [(lw, lh) for lw in range(2, 7) for lh in range(2, 7) if (lw == 6) == (lh == 6)]
CTU = 128
O_NO_MIP = 2                                 # VVCB_VISIT_NO_MIP


def picture(kind, bd, H, W):
    y, x = np.mgrid[0:H, 0:W]
    hi = (1 << bd) - 1
    if kind == 'flat':                       # every prediction equals the original: all distances 0
        orig = np.full((H, W), 1 << (bd - 1))
        reco = orig.copy()
    elif kind == 'offset':                   # flat, original and reconstruction apart: all distances equal, not 0
        orig = np.full((H, W), hi // 3)
        reco = np.full((H, W), 2 * hi // 3)
    elif kind == 'checker':                  # period two in both directions
        orig = np.where((x + y) & 1, hi, 0)
        reco = orig.copy()
    else:                                    # 'stripes': vertical stripes of period four, the reconstruction their mirror
        orig = np.where((x >> 1) & 1, hi, hi // 4)
        reco = np.where((y >> 1) & 1, hi, hi // 4)
    return orig.astype(np.int16), reco.astype(np.int16)


def visits(rng, W, H, n_per_shape):
    out = []
    for lw, lh in SHAPES:
        w, h = 1 << lw, 1 << lh
        for k in range(n_per_shape):
            v = np.zeros(1, O.VISIT_DTYPE)[0]
            v['x'] = 4 * rng.integers(1, (W - 2 * w) // 4)
            on_row = k % 2 == 0                                    # MRL allowed only off a CTU row
            v['y'] = CTU * rng.integers(1, H // CTU) if on_row else 4 * rng.integers(1, (H - 2 * h) // 4) | 4
            v['log2w'], v['log2h'] = lw, lh
            v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = 1, w // 4, w // 4, h // 4, h // 4
            v['flags'] = O_NO_MIP if k % 3 == 2 else 0
            mpm, nc = O.intra_mpms(int(rng.integers(0, 67)), int(rng.integers(0, 67)))
            v['mpm'], v['num_mpm_cand'] = mpm, nc
            # equal rates: equal bits for every non-MPM mode of one binarisation length; a zero lambda: cost == distance
            v['rates'] = np.full(11, 32768) if k % 4 < 2 else rng.integers(100, 200000, 11)
            v['sqrt_lambda'] = 0.0 if k % 4 in (0, 3) else float(rng.uniform(1e-4, 3e-3))
            out.append(v)
    return np.array(out, O.VISIT_DTYPE)


@pytest.mark.parametrize('kind', ['flat', 'offset', 'checker', 'stripes'])
@pytest.mark.parametrize('bd', [8, 10])
def test_lists_on_ties_match_oracle(emul, kind, bd):  # noqa: F811
    rng = np.random.default_rng(1000 * bd + len(kind))
    H, W = 3 * CTU, 512
    orig, reco = picture(kind, bd, H, W)
    arr = visits(rng, W, H, 6)[:-1]          # an odd number of visits: the last CTA of the list kernel is partly empty
    assert len(arr) % 2 == 1
    res, det, _ = run_emul(emul, orig, reco, bd, arr)
    ora, odet = O.rmd_batch(orig, reco, bd, CTU, arr)
    bad = [i for i in range(len(arr)) if res[i].tobytes() != ora[i].tobytes() or det[i].tobytes() != odet[i].tobytes()]
    assert not bad, (len(bad), arr[bad[0]])
    # the lists must be full of ties, or the test says nothing about them
    tied = sum(len(set(r['rd_cost'][:int(r['n_rd'])].tolist())) < int(r['n_rd']) for r in ora)
    assert tied > len(arr) // 2
    # the brief records, from the same distances
    import vvc_intra_b200 as vb
    brief = np.zeros(len(arr), vb.BRIEF_DTYPE)
    assert emul.emul_rmd_brief(arr.ctypes.data_as(C.c_void_p), len(arr), CTU, odet.ctypes.data_as(C.c_void_p), brief.ctypes.data_as(C.c_void_p)) == 0
    assert brief_matches(brief, ora)
