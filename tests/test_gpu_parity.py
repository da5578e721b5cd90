"""GPU parity tests (run on the B200 box with -m gpu): the CUDA path, called through the C ABI, against the
reference encoder's golden records, against the oracle on seeded random inputs, and -- at BASELINE.json's
full 1080p size -- through sampled oracle checks and size-independent properties."""
import numpy as np
import pytest

import vvc_intra_b200 as vb
from oracle import oracle_py as O
import golden_util as G
from make_golden import SERVED_WORKLOADS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng10():
    with vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=128) as e:
        yield e


@pytest.fixture(scope='module')
def eng8():
    with vb.IntraCostEngine(device=0, bit_depth=8, ctu_size=128) as e:
        yield e


@pytest.mark.parametrize('name,bd', [('ref_8b_128x64_qp32', 8), ('ref_10b_192x128_qp27', 10)])
def test_golden_fixture_parity(name, bd, eng8, eng10):
    """Every recorded visit of the reference encoder: SAD/SATD of every evaluation, candidate lists with
    exact double costs, and byte-identical result structs versus the oracle."""
    _check_fixture(name, bd, eng8 if bd == 8 else eng10)


@pytest.mark.parametrize('name', sorted(SERVED_WORKLOADS))
def test_served_workload_visits_match_reference(name, eng8, eng10):
    """The pictures the reference encoder encodes in the served-encoder tests below (tools/make_golden.py SERVED_WORKLOADS), checked without
    the reference binaries: sampled rough-mode-decision visits of the reference against the engine, as in test_golden_fixture_parity."""
    bd = 8 if '_8b_' in name else 10
    _check_fixture('served/' + name, bd, eng8 if bd == 8 else eng10)


def _check_fixture(name, bd, eng):
    visits, _ = G.load_fixture(name)
    orig, reco, arr = G.build_atlas(visits)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    res, det = eng.rmd_eval(arr, detail=True)
    errs = []
    for v, r, d in zip(visits, res, det):
        errs += G.check_visit_against_reference(v, r, d)
    assert not errs, errs[:5]
    ora, odet = O.rmd_batch(orig, reco, bd, 128, arr)
    assert np.array_equal(det['sad'], odet['sad']) and np.array_equal(det['satd'], odet['satd'])
    assert res.tobytes() == ora.tobytes() and det.tobytes() == odet.tobytes()


def test_prediction_samples_match_reference(eng8):
    """Prediction samples (not only their distortion) of the visits recorded with full samples."""
    visits, _ = G.load_fixture('ref_8b_128x64_qp32')
    sel = [v for v in visits if any('pred' in e for e in v['evals'])][:17 * 2]
    orig, reco, arr = G.build_atlas(sel)
    eng8.frame_begin(orig)
    eng8.reco_update(reco)
    n = 0
    for v, a in zip(sel, arr):
        for e in v['evals'][::7]:
            if 'pred' not in e:
                continue
            got = eng8.rmd_pred(a, G.slot_of(v['head'], e))
            assert np.array_equal(got, e['pred']), (v['head']['w'], v['head']['h'], e['mip'], e['mrl'], e['mode'])
            n += 1
    assert n > 100


@pytest.mark.parametrize('bd,seed', [(8, 1), (10, 2), (10, 3)])
def test_random_visits_match_oracle(bd, seed, eng8, eng10):
    """Seeded random planes, random ragged availability, random MPM lists / rates / lambda, all 17 shapes."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, reco, arr = G.random_case(rng, bd, 24)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    res, det = eng.rmd_eval(arr, detail=True)
    ora, odet = O.rmd_batch(orig, reco, bd, 128, arr)
    bad = [i for i in range(len(arr)) if res[i].tobytes() != ora[i].tobytes() or det[i].tobytes() != odet[i].tobytes()]
    assert not bad, (len(bad), arr[bad[0]], [s for s in range(112) if det[bad[0]]['satd'][s] != odet[bad[0]]['satd'][s]])


def test_extreme_sample_values(eng10):
    """All-zero / all-max / checkerboard content: largest residuals the SATD accumulators can see."""
    H, W = 256, 512
    yy, xx = np.mgrid[0:H, 0:W]
    for orig, reco in ((np.zeros((H, W), np.int16), np.full((H, W), 1023, np.int16)),
                       (((xx + yy) % 2 * 1023).astype(np.int16), ((xx + yy + 1) % 2 * 1023).astype(np.int16))):
        rng = np.random.default_rng(7)
        _, _, arr = G.random_case(rng, 10, 3, plane=(H, W))
        eng10.frame_begin(orig)
        eng10.reco_update(reco)
        res, det = eng10.rmd_eval(arr, detail=True)
        ora, odet = O.rmd_batch(orig, reco, 10, 128, arr)
        assert res.tobytes() == ora.tobytes() and det.tobytes() == odet.tobytes()


def test_full_1080p_sweep_properties(eng10):
    """BASELINE config 2 size: every candidate CU of a 1920x1080 10-bit picture (679 260 visits).  Checked by
    (i) ALL visits against the oracle (lists, costs, SAD / SATD of every slot), (ii) determinism, (iii) domain properties: DC-only
    content has zero distortion for planar/DC, list costs ascend, SATD of identical blocks is zero."""
    import sys
    sys.path.insert(0, 'tools')
    from make_golden import synth_yuv
    Y, _, _ = synth_yuv(1920, 1080, 10)
    orig = Y.astype(np.int16)
    vis = vb.build_sweep_visits(1920, 1080, qp=32)
    assert len(vis) == 679260
    eng10.frame_begin(orig)
    eng10.reco_update(orig)            # speculative sweep: neighbours taken from the original picture
    res, det = eng10.rmd_eval(vis, detail=True)
    res2 = eng10.rmd_eval(vis)
    assert res.tobytes() == res2.tobytes()
    # EVERY visit of the frame against the oracle: lists (modes and double costs) and the SAD / SATD of every slot; the oracle is a plain-C
    # loop over visits without shared state, so the host's cores share it (ctypes releases the GIL)
    import os
    from concurrent.futures import ThreadPoolExecutor
    O.rmd_batch(orig, orig, 10, 128, vis[:1])                        # loads the library before the threads start
    parts = np.array_split(np.arange(len(vis)), 8 * (os.cpu_count() or 1))
    def check(ix):
        ora, odet = O.rmd_batch(orig, orig, 10, 128, vis[ix])
        return res[ix].tobytes() == ora.tobytes() and det[ix].tobytes() == odet.tobytes()
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as pool:
        assert all(pool.map(check, parts))
    rng = np.random.default_rng(11)
    idx = np.sort(rng.choice(len(vis), 3000, replace=False))
    n_rd = res['n_rd']
    assert n_rd.min() >= 2 and n_rd.max() <= vb.engine.MAX_LIST
    for i in idx[:200]:
        c = res[i]['had_cost'][:res[i]['n_had']]
        assert np.all(np.diff(c) >= 0)
    # flat picture: planar and DC predict it exactly wherever any neighbour exists
    flat = np.full((1080, 1920), 600, np.int16)
    eng10.frame_begin(flat)
    eng10.reco_update(flat)
    _, d3 = eng10.rmd_eval(vis[:20000], detail=True)
    has_nb = (vis[:20000]['n_above'] > 0) | (vis[:20000]['n_left'] > 0)
    assert np.all(d3['satd'][has_nb][:, :2] == 0) and np.all(d3['sad'][has_nb][:, :2] == 0)


def test_pipeline_chunk_schedule_edges(eng10, tmp_path):
    """The chunked host-buffer path (short first chunk, full chunks, short last chunk) for batch sizes around every boundary of the
    schedule: a child process with VVCB_PIPE_CHUNK=4096 (edge chunks of 1024 visits) must return, for each size, exactly what the
    one-shot path returns here."""
    import hashlib
    import json
    import os
    import subprocess
    import sys
    from make_golden import synth_yuv
    sizes = [4097, 5120, 5121, 8191, 8192, 8193, 9216, 9217, 12289, 20000]
    Y = synth_yuv(416, 240, 10)[0].astype(np.int16)
    vis = vb.build_sweep_visits(416, 240, qp=32)
    assert len(vis) >= max(sizes)
    eng10.frame_begin(Y)
    eng10.reco_update(Y)
    want = {n: hashlib.sha256(eng10.rmd_eval(vis[:n], detail=True)[0].tobytes()).hexdigest() for n in sizes}      # detail => one shot
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child = (
        "import sys, json, hashlib, numpy as np\n"
        "sys.path.insert(0, %r); sys.path.insert(0, %r + '/tools')\n"
        "import vvc_intra_b200 as vb\n"
        "from make_golden import synth_yuv\n"
        "Y = synth_yuv(416, 240, 10)[0].astype(np.int16)\n"
        "vis = vb.build_sweep_visits(416, 240, qp=32)\n"
        "out = {}\n"
        "with vb.IntraCostEngine(0, 10, 128) as eng:\n"
        "    eng.frame_begin(Y); eng.reco_update(Y)\n"
        "    for n in %r:\n"
        "        out[n] = hashlib.sha256(eng.rmd_eval(vis[:n]).tobytes()).hexdigest()\n"
        "print(json.dumps(out))\n" % (root, root, sizes))
    r = subprocess.run([sys.executable, '-c', child], env=dict(os.environ, VVCB_PIPE_CHUNK='4096'), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    got = {int(k): v for k, v in json.loads(r.stdout.strip().splitlines()[-1]).items()}
    assert got == want


def test_error_behaviour(eng10):
    orig = np.zeros((64, 64), np.int16)
    eng10.frame_begin(orig)
    v = np.zeros(1, vb.VISIT_DTYPE)
    v['x'], v['y'], v['log2w'], v['log2h'] = 32, 32, 6, 6      # sticks out of the picture
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.rmd_eval(v)
    v['log2w'], v['log2h'] = 3, 3
    v['n_above'] = 5                                             # more units than the CU is wide
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.rmd_eval(v)
    assert len(eng10.rmd_eval(np.zeros(0, vb.VISIT_DTYPE))) == 0  # empty batch
    with vb.IntraCostEngine(device=0, bit_depth=10) as fresh:
        with pytest.raises(vb.EngineError, match='frame_begin'):
            fresh.rmd_eval(np.zeros(1, vb.VISIT_DTYPE))
    with pytest.raises(vb.EngineError):
        vb.IntraCostEngine(device=99)


# ---- TU coding (vvcb_tu_eval) ---------------------------------------------------------------------------
@pytest.mark.parametrize('name,bd', [('ref_8b_128x64_qp32', 8), ('ref_10b_192x128_qp27', 10), ('ref_10b_64x64_qp32_scalarq', 10)])
def test_tu_golden_parity(name, bd, eng8, eng10):
    """Forward DCT-II / DST-VII / DCT-VIII / transform-skip coefficients and pre-selection sums of the reference's
    transformNxN(trModes) records; levels and uiAbsSum of its Quant::quant records; reconstruction + SSE versus the oracle."""
    eng = eng8 if bd == 8 else eng10
    _, tus = G.load_fixture(name)
    orig, jobs, resi, pred, items = G.build_tu_batch(tus, bd)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True)
    errs = G.check_tu_outputs(items, bd, out)
    assert not errs, errs[:5]
    # the candidate selection of TrQuant::transformNxN(trModes) from the kernel's sums
    k = 0
    while k < len(items):
        if items[k]['kind'] != 'S':
            k += 1
            continue
        r = items[k]['rec']
        m = len(r['modes'])
        sel = eng.mts_preselect(out['results']['abs_sum_coeff'][k:k + m], r['w'], r['h'], r['max_cand'])
        assert list(sel) == [x['selected'] for x in r['modes']]
        k += m


@pytest.mark.parametrize('bd,seed', [(8, 31), (10, 32), (10, 33)])
def test_tu_random_blocks_match_oracle(bd, seed, eng8, eng10):
    """Every (shape, transform) incl. 64-point sides with their zero-out, random QP, small to full-range residuals."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, jobs, resi, pred, items = G.random_tu_case(rng, bd, 3)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True)
    exp = G.oracle_tu_chain(items, bd)
    for k in ('coeff', 'level', 'reco'):
        assert np.array_equal(out[k], exp[k]), k
    assert out['results'].tobytes() == exp['results'].tobytes()
    # properties: a zero residual quantises to nothing and reconstructs the prediction
    z = eng.tu_eval(jobs, np.zeros_like(resi), pred, want_level=True, want_reco=True)
    assert not z['level'].any() and np.array_equal(z['reco'], pred) and not z['results']['abs_sum_coeff'].any()


def test_tu_error_behaviour(eng10):
    eng10.frame_begin(np.zeros((64, 64), np.int16))
    j = np.zeros(1, vb.TU_JOB_DTYPE)
    j['log2w'], j['log2h'], j['mts_idx'] = 6, 6, 2              # MTS is not allowed on 64-point sides
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.tu_eval(j, np.zeros(4096, np.int16))
    j['mts_idx'], j['flags'] = 0, vb.TU_QUANT
    with pytest.raises(vb.EngineError, match='prediction'):
        eng10.tu_eval(j, np.zeros(4096, np.int16))


# ---- texture measures (vvcb_ctu_hads_islice, vvcb_features_eval) ------------------------------------------
def test_ctu_hads_islice_parity(eng10):
    """EncCu::updateCtuDataISlice: the reference's own per-CTU sums (ragged 72-wide / 8-high CTUs), then a 1080p frame."""
    _, recs = G.load_fixture('ref_10b_200x136_ctuhad')
    hs = [r for r in recs if r['tag'] == 'H']
    pic = np.zeros((136, 200), np.int16)
    pic[:128, :128], pic[:128, 128:], pic[128:, :128], pic[128:, 128:] = [r['org'] for r in hs]
    eng10.frame_begin(pic)
    assert eng10.ctu_hads_islice(200, 136).tolist() == [r['result'] for r in hs]
    from make_golden import synth_yuv
    Y = synth_yuv(1920, 1080, 10)[0].astype(np.int16)
    eng10.frame_begin(Y)
    got = eng10.ctu_hads_islice(1920, 1080)
    assert got.shape == (135,) and got.tolist() == O.ctu_hads_islice(Y, ctu=128).tolist()
    eng10.frame_begin(np.full((64, 64), 513, np.int16))       # flat content has no AC energy
    assert eng10.ctu_hads_islice(64, 64).tolist() == [0]
    with pytest.raises(vb.EngineError, match='CTUs'):
        eng10._ck(eng10._lib.vvcb_ctu_hads_islice(eng10._ctx, np.zeros(3, np.int32).ctypes.data, 3))


@pytest.mark.parametrize('seed,mx', [(51, 256), (52, 1024), (53, 40)])
def test_features_match_oracle(seed, mx, eng10):
    """FAST_ALGORITHM features on random content (8-bit range, 10-bit range saturating to 255 as the reference does,
    and a low-contrast picture with many rounding ties), random CU shapes and neighbour sets."""
    from test_oracle_features import random_feature_jobs
    rng = np.random.default_rng(seed)
    H, W = 256, 512
    pic = rng.integers(0, mx, (H, W)).astype(np.int16)
    pic[:, 256:] = (pic[:, 256:] // 8) * 8 % 256
    jobs = random_feature_jobs(rng, H, W, 3000)
    eng10.frame_begin(pic)
    got = eng10.features_eval(jobs)
    exp = O.features_batch(pic, jobs)
    bad = [i for i in range(len(jobs)) if got[i].tobytes() != exp[i].tobytes()]
    assert not bad, (len(bad), jobs[bad[0]]['cu'], got[bad[0]]['f'].tolist(), exp[bad[0]]['f'].tolist())


def test_features_on_a_partitioned_picture(eng10):
    """Config 4 shape of use: every CU of a random QT/MTT partition of a 416x240 picture, neighbours picked by the
    host logic (vvc_intra_b200.features), checked against the oracle; plus the error behaviour."""
    from test_host_features import random_partition, cu_lookup
    from make_golden import synth_yuv
    Y = synth_yuv(416, 240, 8)[0].astype(np.int16)
    rng = np.random.default_rng(5)
    cus = random_partition(rng, 416, 240)
    get_cu = cu_lookup(cus, 416, 240)
    jobs = []
    for c in cus:
        if vb.feature_gate(c['x'], c['y'], c['w'], c['h'], c['mt_depth']):
            jobs.append(vb.feature_job(c['x'], c['y'], c['w'], c['h'], c['qt_depth'], c['mt_depth'],
                                       vb.select_feature_neighbours(get_cu, c['x'], c['y'], c['w'], c['h'])))
    jobs = np.array(jobs, vb.FEAT_JOB_DTYPE)
    assert len(jobs) > 100
    eng10.frame_begin(Y)
    got = eng10.features_eval(jobs)
    assert got.tobytes() == O.features_batch(Y, jobs).tobytes()
    assert got['valid'].sum() > 50
    bad = jobs[:1].copy()
    bad['cu']['w'] = 12
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.features_eval(bad)
    assert len(eng10.features_eval(jobs[:0])) == 0


def test_features_full_1080p_sweep(eng10):
    """Config 4 at its stated size: the features of every candidate CU of a 1920x1080 10-bit frame (549 660 jobs, 10-bit content
    saturating to 255 as the reference's convertTo(CV_8U) does).  Every 97th job against the oracle; size-independent properties on
    all of them: f0..f3 echo the job, valid <=> at least three neighbours, and a CU of a flat picture has zero gradients and variances."""
    from make_golden import synth_yuv
    from vvc_intra_b200.features import build_sweep_feature_jobs
    Y = synth_yuv(1920, 1080, 10)[0].astype(np.int16)
    jobs = build_sweep_feature_jobs(1920, 1080)
    assert len(jobs) == 549660
    eng10.frame_begin(Y)
    got = eng10.features_eval(jobs)
    sel = slice(None, None, 97)
    assert got[sel].tobytes() == O.features_batch(Y, jobs[sel]).tobytes()
    assert np.array_equal(got['f'][:, 0], jobs['cu']['h']) and np.array_equal(got['f'][:, 1], jobs['cu']['w'])
    assert np.array_equal(got['f'][:, 2], jobs['cu']['qt_depth']) and np.array_equal(got['f'][:, 3], jobs['cu']['mt_depth'])
    assert np.array_equal(got['valid'] != 0, jobs['n_neighbours'] >= 3)
    flat = np.full_like(Y, 130)
    eng10.frame_begin(flat)
    gf = eng10.features_eval(jobs[::11])
    v = gf['valid'] != 0
    assert v.sum() > 1000 and not gf['f'][v][:, 4:12].any() and not gf['f'][v][:, 21:26].any()


# ---- dependent quantisation (VVCB_TU_DEPQUANT) -----------------------------------------------------------
@pytest.mark.parametrize('name,bd', [('ref_10b_128x128_qp27_depquant', 10), ('ref_8b_128x64_qp37_depquant', 8)])
def test_dep_quant_golden_parity(name, bd, eng8, eng10):
    """DQIntern::DepQuant::quant as the reference ran it: recorded residuals and context prices in, the recorded
    coefficients, levels and absSum out; reconstruction + SSE versus the oracle's state-machine dequantiser."""
    eng = eng8 if bd == 8 else eng10
    _, tus = G.load_fixture(name)
    orig, jobs, resi, pred, rates, items = G.build_dq_batch(tus, bd)
    assert len(items) > 80
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates)
    errs = G.check_dq_outputs(items, bd, out)
    assert not errs, (len(errs), errs[:6])


@pytest.mark.parametrize('bd,seed', [(8, 71), (10, 72), (10, 73)])
def test_dep_quant_random_blocks_match_oracle(bd, seed, eng8, eng10):
    """Every shape x transform, random QP / lambda / context prices / LFNST first-position rule, mixed with scalar-quantiser
    jobs in the same batch (the two quantisers share the transform and reconstruction passes)."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, jobs, resi, pred, rates, items = G.random_dq_case(rng, bd, 4)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates)
    exp = G.oracle_dq_chain(items, bd)
    for k in ('coeff', 'level', 'reco'):
        bad = [i for i, it in enumerate(items) if not np.array_equal(out[k][it['off']:it['off'] + it['resi'].size], exp[k][it['off']:it['off'] + it['resi'].size])]
        assert not bad, (k, len(bad), [(items[i]['resi'].shape, items[i]['mts'], items[i]['qp'], items[i]['lfnst']) for i in bad[:5]])
    assert out['results'].tobytes() == exp['results'].tobytes()
    assert (out['results']['abs_sum_level'] > 0).sum() > len(items) // 3
    # half of the jobs switched to the scalar quantiser: both kinds in one call
    mixed = jobs.copy()
    mixed['flags'][::2] = vb.TU_QUANT
    out2 = eng.tu_eval(mixed, resi, pred, want_level=True, want_reco=True, rates=rates)
    for i, it in enumerate(items):
        sl = slice(it['off'], it['off'] + it['resi'].size)
        if i % 2:
            assert np.array_equal(out2['level'][sl], exp['level'][sl]) and out2['results'][i].tobytes() == exp['results'][i].tobytes()
        else:
            h, w = it['resi'].shape
            lvl, s = O.quant_scalar(exp['coeff'][sl].reshape(h, w), bd, it['qp'] // 6, it['qp'] % 6, False)
            assert np.array_equal(out2['level'][sl].reshape(h, w), lvl) and int(out2['results'][i]['abs_sum_level']) == s
    # deterministic
    out3 = eng.tu_eval(jobs, resi, pred, want_level=True, rates=rates)
    assert np.array_equal(out3['level'], out['level'])


def test_dep_quant_error_behaviour(eng10):
    eng10.frame_begin(np.zeros((64, 64), np.int16))
    j = np.zeros(1, vb.TU_JOB_DTYPE)
    j['log2w'], j['log2h'], j['flags'], j['lambda'] = 3, 3, vb.TU_QUANT | vb.TU_DEPQUANT, 10.0
    z = np.zeros(64, np.int16)
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.tu_eval(j, z, z)                                     # no context prices
    j['mts_idx'] = 1
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.tu_eval(j, z, z, rates=np.zeros(1, vb.DQ_RATES_DTYPE))   # transform skip is not dependent-quantised
    j['mts_idx'] = 0
    out = eng10.tu_eval(j, z, z, want_level=True, want_reco=True, rates=np.zeros(1, vb.DQ_RATES_DTYPE))
    assert not out['level'].any() and out['results']['abs_sum_level'][0] == 0 and out['results']['sse'][0] == 0


# ---- xIntraCodingTUBlock as a whole (vvcb_tu_eval_pred) -----------------------------------------------------
@pytest.mark.parametrize('bd,seed', [(8, 91), (10, 92)])
def test_tu_eval_with_device_prediction(bd, seed, eng8, eng10):
    """Prediction (regular, MRL and MIP slots, ragged availability) -> residual -> transform -> dependent quantisation ->
    reconstruction -> SSE, all on the device from the frame planes; every stage against the oracle."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, reco, visits, src, jobs, n_samples, rates, items = G.pred_tu_case(rng, bd, 6)
    eng.frame_begin(orig)
    eng.reco_update(reco)
    out = eng.tu_eval_pred(visits, src, jobs, n_samples, want_coeff=True, want_level=True, want_reco=True, want_pred=True, rates=rates)
    exp = G.oracle_dq_chain(items, bd)
    for i, it in enumerate(items):
        sl = slice(it['off'], it['off'] + it['pred'].size)
        assert np.array_equal(out['pred'][sl].reshape(it['pred'].shape), it['pred']), (i, it['pred'].shape, int(src[i]['slot']))
    for k in ('coeff', 'level', 'reco'):
        assert np.array_equal(out[k], exp[k]), k
    assert out['results'].tobytes() == exp['results'].tobytes()
    # the same jobs through the host-buffer entry point give the same answer
    resi = np.concatenate([it['resi'].ravel() for it in items])
    pred = np.concatenate([it['pred'].ravel() for it in items])
    out2 = eng.tu_eval(jobs, resi, pred, want_level=True, want_reco=True, rates=rates)
    assert np.array_equal(out2['level'], out['level']) and np.array_equal(out2['reco'], out['reco']) and out2['results'].tobytes() == out['results'].tobytes()
    # error behaviour: a slot the visit does not evaluate, a job whose geometry is not the visit's
    bad = src.copy()
    bad['slot'][0] = 200
    with pytest.raises(vb.EngineError, match='malformed'):
        eng.tu_eval_pred(visits, bad, jobs, n_samples, rates=rates)
    badj = jobs.copy()
    badj['x'][0] += 4
    with pytest.raises(vb.EngineError, match='malformed'):
        eng.tu_eval_pred(visits, src, badj, n_samples, rates=rates)


# ---- RDOQ of transform-skip TUs (VVCB_TU_RDOQ_TS) -----------------------------------------------------------
@pytest.mark.parametrize('name,bd', [('ref_10b_128x128_qp27_rdoqts', 10), ('ref_8b_128x64_qp37_rdoqts', 8)])
def test_rdoq_ts_golden_parity(name, bd, eng8, eng10):
    """QuantRDOQ::xRateDistOptQuantTS as the reference ran it (RDOQTS on as shipped): recorded residuals and context prices in,
    the recorded levels and absSum out; reconstruction + SSE versus the oracle."""
    eng = eng8 if bd == 8 else eng10
    _, tus = G.load_fixture(name)
    orig, jobs, resi, pred, rates, items = G.build_rdoq_batch(tus, bd)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates)
    errs = G.check_rdoq_outputs(items, bd, out)
    assert not errs, (len(errs), errs[:6])


@pytest.mark.parametrize('bd,seed', [(8, 111), (10, 112)])
def test_rdoq_ts_random_blocks_match_oracle(bd, seed, eng8, eng10):
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, jobs, resi, pred, rates, items = G.random_rdoq_case(rng, bd, 12)
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates)
    exp = G.oracle_rdoq_chain(items, bd)
    for k in ('coeff', 'level', 'reco'):
        assert np.array_equal(out[k], exp[k]), k
    assert out['results'].tobytes() == exp['results'].tobytes()
    bad = jobs[:1].copy()
    bad['mts_idx'] = 0                                       # RDOQ_TS is for transform skip only
    with pytest.raises(vb.EngineError, match='malformed'):
        eng.tu_eval(bad, resi, pred, rates=rates)


# ---- LFNST (cu.lfnstIdx 1 / 2) ---------------------------------------------------------------------------------
@pytest.mark.parametrize('name,bd', [('ref_10b_128x128_qp27_lfnst', 10), ('ref_8b_128x64_qp32_lfnst', 8)])
def test_lfnst_golden_parity(name, bd, eng8, eng10):
    """TrQuant::xFwdLfnst / xInvLfnst around the dependent quantiser as the reference ran them: coefficients of the LFNST region,
    levels, absSum from the 'F' records; reconstruction + SSE versus the oracle chain (inverse half pinned by the 'J' records)."""
    eng = eng8 if bd == 8 else eng10
    _, tus = G.load_fixture(name)
    orig, jobs, resi, pred, rates, items = G.build_dq_batch(tus, bd, tag='F')
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_coeff=True, want_level=True, want_reco=True, rates=rates)
    errs = G.check_dq_outputs(items, bd, out)
    assert not errs, (len(errs), errs[:6])
    # the scalar quantiser with LFNST: same coefficients, levels of Quant::quant on them (oracle)
    sc = jobs.copy()
    sc['flags'] = vb.TU_QUANT
    out2 = eng.tu_eval(sc, resi, pred, want_coeff=True, want_level=True, want_reco=True)
    assert np.array_equal(out2['coeff'], out['coeff'])
    for i, it in enumerate(items[:40]):
        r = it['rec']
        h, w = r['resi'].shape
        sl = slice(it['off'], it['off'] + w * h)
        lvl, s = O.quant_scalar(out['coeff'][sl].reshape(h, w), bd, r['per'], r['rem'], False)
        assert np.array_equal(out2['level'][sl].reshape(h, w), lvl)
        res = O.inv_transform(O.inv_lfnst(O.dequant(lvl, bd, r['per'], r['rem'], False), r['intra_mode'], r['lfnst']), bd, r['mts'])
        reco, sse = O.reconstruct_sse(it['org'], it['pred'], res, bd)
        assert np.array_equal(out2['reco'][sl].reshape(h, w), reco) and int(out2['results'][i]['sse']) == int(sse)


# ---- full-size runs of the later stages ---------------------------------------------------------------------
def test_full_1080p_tu_stage_properties(eng10):
    """BASELINE config 2 size for the second stage: the best RMD candidate of every candidate CU of a 1920x1080 10-bit picture
    (679 260 TUs) through vvcb_tu_eval_pred.  Checked by (i) a seeded sample against the oracle chain, (ii) determinism,
    (iii) size-independent properties: SSE equals the host-side sum of squared differences of the returned reconstruction,
    a zero level block reconstructs the prediction, abs sums equal the sums of the returned levels."""
    from make_golden import synth_yuv
    Y = synth_yuv(1920, 1080, 10)[0].astype(np.int16)
    vis = vb.build_sweep_visits(1920, 1080, qp=32)
    eng10.frame_begin(Y)
    eng10.reco_update(Y)
    res = eng10.rmd_eval(vis)
    src, jobs, n_samples, rates = vb.build_tu_jobs_from_lists(vis, res, 32, 10)
    assert len(jobs) == 679260
    out = eng10.tu_eval_pred(vis, src, jobs, n_samples, want_level=True, want_reco=True, want_pred=True, rates=rates)
    out2 = eng10.tu_eval_pred(vis, src, jobs, n_samples, want_level=True, rates=rates)
    assert np.array_equal(out['level'], out2['level']) and out['results'].tobytes() == out2['results'].tobytes()
    r = out['results']
    rng = np.random.default_rng(17)
    idx = np.sort(rng.choice(len(jobs), 400, replace=False))
    _, _, preds = O.rmd_batch(Y, Y, 10, 128, vis[idx], want_pred=True)
    for k, i in enumerate(idx):
        j = jobs[i]
        w, h = 1 << int(j['log2w']), 1 << int(j['log2h'])
        sl = slice(int(j['offset']), int(j['offset']) + w * h)
        p = preds[k][int(src[i]['slot'])]
        assert np.array_equal(out['pred'][sl].reshape(h, w), p)
        org = Y[int(j['y']):int(j['y']) + h, int(j['x']):int(j['x']) + w]
        qp = 6 * int(j['qp_per']) + int(j['qp_rem'])
        co = O.fwd_transform((org.astype(np.int32) - p).astype(np.int16), 10, 0)
        lvl, s = O.dep_quant(co, 10, 0, 0, qp, float(j['lambda']), rates[0], 0)
        assert np.array_equal(out['level'][sl].reshape(h, w), lvl) and int(r[i]['abs_sum_level']) == s
        reco, sse = O.reconstruct_sse(org, p, O.inv_transform(O.dep_dequant(lvl, 10, qp), 10, 0), 10)
        assert np.array_equal(out['reco'][sl].reshape(h, w), reco) and int(r[i]['sse']) == int(sse)
    # properties over every TU, vectorised per shape
    abs_levels = np.abs(out['level'])
    sizes = (1 << jobs['log2w'].astype(np.int64)) * (1 << jobs['log2h'].astype(np.int64))
    ends = np.cumsum(sizes)
    csum = np.concatenate([[0], np.cumsum(abs_levels, dtype=np.int64)])
    assert np.array_equal(csum[ends] - csum[ends - sizes], r['abs_sum_level'].astype(np.int64))
    for lw in range(2, 7):
        for lh in range(2, 7):
            sel = np.nonzero((jobs['log2w'] == lw) & (jobs['log2h'] == lh))[0][:4000]
            if not len(sel):
                continue
            w, h = 1 << lw, 1 << lh
            pos = jobs['offset'][sel].astype(np.int64)[:, None] + np.arange(w * h)[None, :]
            yy = jobs['y'][sel].astype(np.int64)[:, None, None] + np.arange(h)[None, :, None]
            xx = jobs['x'][sel].astype(np.int64)[:, None, None] + np.arange(w)[None, None, :]
            org = Y[yy, xx].reshape(len(sel), -1).astype(np.int64)
            rec = out['reco'][pos].astype(np.int64)
            assert np.array_equal(((org - rec) ** 2).sum(axis=1), r['sse'][sel].astype(np.int64))
            zero = r['abs_sum_level'][sel] == 0
            assert np.array_equal(rec[zero], out['pred'][pos][zero].astype(np.int64))


def test_2160p_sweep_properties(eng10):
    """BASELINE config 3 picture size (3840x2160 10-bit, 2 720 940 visits in one call): sampled visits against the oracle,
    the chunked host pipeline against itself, and the list invariants."""
    from make_golden import synth_yuv
    Y = synth_yuv(3840, 2160, 10)[0].astype(np.int16)
    vis = vb.build_sweep_visits(3840, 2160, qp=27)
    assert len(vis) == 2720940          # 30 x 17 CTUs; the bottom CTU row is 112 luma rows high, candidates below the picture are dropped
    eng10.frame_begin(Y)
    eng10.reco_update(Y)
    res = eng10.rmd_eval(vis)
    assert res['n_rd'].min() >= 2 and res['n_final'].max() <= vb.engine.MAX_LIST and (res['n_final'] >= res['n_rd']).all()
    rng = np.random.default_rng(23)
    idx = np.sort(rng.choice(len(vis), 1500, replace=False))
    ora, _ = O.rmd_batch(Y, Y, 10, 128, vis[idx])
    assert res[idx].tobytes() == ora.tobytes()
    res2 = eng10.rmd_eval(vis[:300000])
    assert res2.tobytes() == res[:300000].tobytes()


# ---- residual rate estimation (vvcb_residual_bits, VVCB_TU_RATE) --------------------------------------------
@pytest.mark.parametrize('name', ['ref_10b_128x128_qp27_resbits', 'ref_8b_128x64_qp22_resbits'])
def test_residual_bits_golden_parity(name, eng10):
    """CABACWriter::residual_coding on the reference's bit estimator: recorded levels and context states in, the fractional bits the
    call added out (regular, MTS and transform-skip residual coding)."""
    _, tus = G.load_fixture(name)
    jobs, levels, states, recs = G.build_rate_batch(tus)
    got = eng10.residual_bits(jobs, levels, states)
    bad = [(r['w'], r['h'], r['mts'], int(g), r['bits']) for g, r in zip(got, recs) if int(g) != r['bits']]
    assert not bad, (len(bad), bad[:5])
    assert eng10.residual_bits(jobs, np.zeros_like(levels), states).max() == 0        # nothing to code
    eng10.set_option(vb.OPT_DEP_QUANT, 0)                                             # without the quantiser state machine: set 0 always
    try:
        alt = eng10.residual_bits(jobs, levels, states)
        exp = [O.residual_bits(r['level'], r['mts'], r['ts_allowed'], r['mts_allowed'], 0, O.ctx_states_from_record(r['states'])) for r in recs]
        assert alt.tolist() == exp and alt.tolist() != got.tolist()
    finally:
        eng10.set_option(vb.OPT_DEP_QUANT, 1)


@pytest.mark.parametrize('bd,seed', [(8, 121), (10, 122)])
def test_tu_stage_returns_residual_bits(bd, seed, eng8, eng10):
    """VVCB_TU_RATE inside the TU pipeline: the bits of the levels the quantisers just produced (dependent quantisation with and without
    LFNST / MTS, transform-skip RDOQ), against the oracle pricing the oracle's levels."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    orig, jobs, resi, pred, rates, items = G.random_dq_case(rng, bd, 2)
    states = np.zeros(len(rates), vb.CTX_STATES_DTYPE)
    flat = states.view(vb.BIN_MODEL_DTYPE).reshape(len(rates), -1)
    flat['state'][..., 0] = rng.integers(1, 1023, flat.shape) << 5                  # MASK_0 domain
    flat['state'][..., 1] = rng.integers(1, 16383, flat.shape) << 1                 # MASK_1 domain
    flat['rate'] = (rng.integers(4, 8, flat.shape) << 4) | rng.integers(4, 10, flat.shape)
    jobs = jobs.copy()
    jobs['flags'] |= vb.TU_RATE | vb.TU_TS_ALLOWED
    jobs['flags'][(jobs['log2w'] <= 5) & (jobs['log2h'] <= 5)] |= vb.TU_MTS_ALLOWED
    for it, j in zip(items, jobs):
        it['bits_fn'] = (lambda lv, j=j: O.residual_bits(lv, int(j['mts_idx']), True, bool(j['flags'] & vb.TU_MTS_ALLOWED), 1, states[int(j['rate_idx'])]))
    eng.frame_begin(orig)
    out = eng.tu_eval(jobs, resi, pred, want_level=True, rates=rates, states=states)
    exp = G.oracle_dq_chain(items, bd)
    assert np.array_equal(out['level'], exp['level'])
    assert out['results'].tobytes() == exp['results'].tobytes()
    assert (out['results']['frac_bits'] > 0).sum() > len(items) // 3
    # the stand-alone entry point on the same levels
    assert eng.residual_bits(jobs, out['level'], states).tolist() == out['results']['frac_bits'].tolist()


# ---- the unmodified reference encoder with the engine plugged in ---------------------------------------------
@pytest.mark.parametrize('w,h,bits,qp', [(128, 64, 8, 32), (128, 128, 10, 27)])
def test_reference_encoder_with_gpu_rmd_is_bit_identical(w, h, bits, qp, tmp_path):
    """Drop-in check at the reference's own seam: oracle/_ref/EncoderAppGpu is the unmodified reference encoder linked (ld --wrap,
    oracle/ref_gpu_shim.cpp) so that every rough-mode-decision prediction comes from libvvc_intra_b200.so and every candidate list the
    reference builds is compared with vvcb_rmd_eval's; every luma TU (no ISP) is transformed, pre-selected, quantised (dependent quantisation,
    transform-skip RDOQ, LFNST) and reconstructed by vvcb_tu_eval and priced by vvcb_residual_bits next to the reference, the encoder going
    on with the engine's levels.  The shim aborts on the first difference; the bitstream must be byte-identical to the plain reference
    encoder's."""
    import json
    import os
    import subprocess
    from make_golden import synth_yuv
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    plain, plugged, cfg = (os.path.join(root, 'oracle/_ref', f) for f in ('EncoderApp', 'EncoderAppGpu', 'encoder_intra.cfg'))
    if not all(os.path.exists(p) for p in (plain, plugged, cfg)):
        pytest.skip('oracle/_ref binaries are built only in the container that has /root/reference')
    Y, U, V = synth_yuv(w, h, bits)
    (tmp_path / 'in.yuv').write_bytes(Y.tobytes() + U.tobytes() + V.tobytes())
    (tmp_path / 'Time_python.dat').write_bytes(b'')
    args = ['-c', cfg, '-i', 'in.yuv', '-wdt', str(w), '-hgt', str(h), '-q', str(qp), '-f', '1', '-fr', '30',
            '--InputBitDepth=%d' % bits, '--InternalBitDepth=%d' % bits, '--OutputBitDepth=%d' % bits]
    env = dict(os.environ, VVCB_SHIM_REPORT=str(tmp_path / 'report.json'))
    r1 = subprocess.run([plain] + args + ['-b', 'plain.bin'], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r1.returncode == 0, r1.stdout[-2000:]
    r2 = subprocess.run([plugged] + args + ['-b', 'gpu.bin'], cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r2.returncode == 0, r2.stdout[-2000:]
    a, b = (tmp_path / 'plain.bin').read_bytes(), (tmp_path / 'gpu.bin').read_bytes()
    assert len(a) > 100 and a == b
    rep = json.loads((tmp_path / 'report.json').read_text())
    assert rep['mismatches'] == 0 and rep['visits'] > 200 and rep['lists_compared'] == rep['visits'] and rep['predictions_replaced'] > 40 * rep['visits']
    assert rep['tu_quantised'] > 1000 and rep['tu_dep_quant'] > 500 and rep['tu_rdoq_ts'] > 50 and rep['tu_lfnst'] > 100
    assert rep['tu_preselections'] > 200 and rep['tu_preselection_candidates'] >= 2 * rep['tu_preselections']
    assert rep['tu_reconstructions'] > 500 and rep['tu_residual_bits'] > 500
    print('shim report', rep)


# ---- one round trip per CU: vvcb_cu_eval over several pictures of one plane -------------------------------------------------
@pytest.mark.parametrize('bd,seed', [(8, 131), (10, 132)])
def test_cu_eval_merges_independent_requests(bd, seed, eng8, eng10):
    """vvcb_cu_eval with requests that belong to three pictures lying side by side in one plane (what the broker does): rectangles pushed
    with the request, rough mode decision and TU candidates in one call; every output equals the oracle run on each picture alone, and
    equals the separate entry points (vvcb_reco_update_rects + vvcb_rmd_eval + vvcb_tu_eval_pred)."""
    eng = eng8 if bd == 8 else eng10
    rng = np.random.default_rng(seed)
    cell = (256, 512)
    pics = [G.pred_tu_case(np.random.default_rng(seed * 10 + k), bd, 2, slots_per_visit=3) for k in range(3)]
    eng.frame_alloc(3 * cell[1], cell[0])
    reqs, expect = [], []
    for k, (orig, reco, visits, src, jobs, n_samples, rates, items) in enumerate(pics):
        ox = k * cell[1]
        eng.orig_update(orig, ox, 0)
        res, det = O.rmd_batch(orig, reco, bd, 128, visits)
        states = np.zeros(1, vb.CTX_STATES_DTYPE)
        for vi, v in enumerate(visits):
            w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
            x, y = int(v['x']), int(v['y'])
            # the reconstructed neighbourhood of this CU: 4 rows above, 4 columns left (what the shim pushes)
            rects, samples = [], []
            for (rx, ry, rw, rh) in ((max(0, x - 4), y - 4, min(cell[1], x + 2 * w + 4) - max(0, x - 4), 4), (x - 4, y, 4, min(cell[0], y + 2 * h + 4) - y)):
                rects.append((rx + ox, ry, rw, rh, sum(len(s) for s in samples)))
                samples.append(reco[ry:ry + rh, rx:rx + rw].ravel())
            mine = [i for i in range(len(jobs)) if int(src[i]['visit']) == vi]
            jb = jobs[mine].copy()
            jb['x'] += ox
            jb['offset'] = np.arange(len(mine)) * w * h
            jb['rate_idx'] = 0
            vv = visits[vi:vi + 1].copy()
            vv['x'] += ox
            # one snapshot per request: take the first job's
            rate_of = [int(jobs[i]['rate_idx']) for i in mine]
            keep = [i for i, r in zip(mine, rate_of) if r == rate_of[0]] if mine else []
            sel = [mine.index(i) for i in keep]
            reqs.append(dict(rects=np.array(rects, vb.RECT_DTYPE), rect_samples=np.concatenate(samples), visit=vv, want_rmd=vi % 2 == 0,
                             jobs=jb[sel] if keep else None, slots=src['slot'][keep] if keep else None, rates=rates[rate_of[0]:rate_of[0] + 1] if keep else None, states=states))
            if keep:
                reqs[-1]['jobs']['offset'] = np.arange(len(keep)) * w * h
            expect.append((res[vi], det[vi], [items[i] for i in keep]))
    order = rng.permutation(len(reqs))
    ns0, calls0 = eng.cu_eval_phases()
    outs = eng.cu_eval([reqs[i] for i in order])
    ns1, calls1 = eng.cu_eval_phases()
    assert calls1 == calls0 + 1 and all(b >= a for a, b in zip(ns0, ns1)) and ns1[6] > ns0[6] and ns1[7] > ns0[7]      # both device spans were clocked
    # the same batch with the timed-sleep wait (what the broker's workers use) and with the blocking event: identical bytes
    for mode in (20, 1, 0):
        eng.set_option(vb.OPT_YIELD_SYNC, mode)
        again = eng.cu_eval([reqs[i] for i in order])
        for a, b in zip(outs, again):
            assert sorted(a.keys()) == sorted(b.keys()) and all(np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes() for k in a)
    n_rmd = n_tu = 0
    for o, i in zip(outs, order):
        res, det, its = expect[i]
        if reqs[i]['want_rmd']:
            assert o['result'][0].tobytes() == res.tobytes() and o['detail'][0].tobytes() == det.tobytes()
            n_rmd += 1
        if its:
            exp = G.oracle_dq_chain([dict(it, off=k * it['pred'].size) for k, it in enumerate(its)], bd)
            assert np.array_equal(o['level'], exp['level']) and np.array_equal(o['reco'], exp['reco'])
            assert np.array_equal(o['pred'], np.concatenate([it['pred'].ravel() for it in its]))
            assert o['tu_results'].tobytes() == exp['results'].tobytes()
            n_tu += len(its)
    assert n_rmd > 10 and n_tu > 30
    # error behaviour: a job that points outside its request's arrays, a rectangle outside the plane
    bad = dict(reqs[order[0]])
    if bad['jobs'] is not None:
        bad['jobs'] = bad['jobs'].copy()
        bad['jobs']['offset'][0] = 1 << 20
        with pytest.raises(vb.EngineError, match='malformed'):
            eng.cu_eval([bad])
    bad = dict(reqs[order[0]])
    bad['rects'] = bad['rects'].copy()
    bad['rects']['x'][0] = 3 * cell[1] - 2
    with pytest.raises(vb.EngineError, match='malformed|outside'):
        eng.cu_eval([bad])


def _encoder_args(cfg, w, h, bits, qp):
    return ['-c', cfg, '-i', 'in.yuv', '-wdt', str(w), '-hgt', str(h), '-q', str(qp), '-f', '1', '-fr', '30',
            '--InputBitDepth=%d' % bits, '--InternalBitDepth=%d' % bits, '--OutputBitDepth=%d' % bits]


def _ref_binaries(*names):
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    paths = [os.path.join(root, 'oracle/_ref', f) for f in names] + [os.path.join(root, 'oracle/_ref/encoder_intra.cfg')]
    if not all(os.path.exists(p) for p in paths):
        pytest.skip('oracle/_ref binaries are built only in the container that has /root/reference')
    return root, paths


@pytest.mark.parametrize('w,h,bits,qp', [(128, 64, 8, 32), (128, 128, 10, 27), (128, 128, 10, 37)])
def test_reference_encoder_served_by_the_engine_is_bit_identical(w, h, bits, qp, tmp_path):
    """oracle/_ref/EncoderAppServe: the unmodified reference encoder whose luma intra cost evaluation inside estIntraPredLumaQT is SERVED by
    libvvc_intra_b200.so (oracle/ref_gpu_serve.cpp): no reference prediction, SAD / SATD, transform, quantiser, reconstruction, SSE or
    residual pricing runs for a whole-CU luma TU.  Same bitstream as the plain encoder, byte for byte."""
    import json
    import os
    import subprocess
    from make_golden import synth_yuv
    root, (plain, served, cfg) = _ref_binaries('EncoderApp', 'EncoderAppServe')
    Y, U, V = synth_yuv(w, h, bits)
    (tmp_path / 'in.yuv').write_bytes(Y.tobytes() + U.tobytes() + V.tobytes())
    (tmp_path / 'Time_python.dat').write_bytes(b'')
    env = dict(os.environ, VVCB_SHIM_REPORT=str(tmp_path / 'report.json'))
    env.pop('VVCB_BROKER', None)
    env.pop('LD_LIBRARY_PATH', None)
    r1 = subprocess.run([plain] + _encoder_args(cfg, w, h, bits, qp) + ['-b', 'plain.bin'], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r1.returncode == 0, r1.stdout[-2000:]
    r2 = subprocess.run([served] + _encoder_args(cfg, w, h, bits, qp) + ['-b', 'gpu.bin'], cwd=tmp_path, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r2.returncode == 0, r2.stdout[-2000:]
    a, b = (tmp_path / 'plain.bin').read_bytes(), (tmp_path / 'gpu.bin').read_bytes()
    assert len(a) > 100 and a == b
    rep = json.loads((tmp_path / 'report.json').read_text())
    assert rep['enabled'] == 1 and rep['visits'] > 1000 and rep['demand_round_trips'] == 0 and rep['stale_context'] == 0
    assert rep['distortions_served'] == 2 * rep['predictions_skipped'] and rep['tu_quantised'] > 10000 and rep['tu_sse'] == rep['tu_quantised']
    assert rep['tu_residual_bits'] > 5000 and rep['tu_residual_bits_reference'] == 0
    print('serve report', rep)


def test_broker_serves_several_encoders_bit_identically(tmp_path):
    """Four encoder processes (different pictures, QP 22 / 27 / 32 / 37, 10 bit) share ONE engine context through the broker
    (vvc_intra_b200/vvcb_broker): bitstreams byte-identical to the plain encoder's, requests of different clients merged into engine batches."""
    import json
    import os
    import subprocess
    from make_golden import synth_yuv
    root, (plain, served, cfg) = _ref_binaries('EncoderApp', 'EncoderAppServe')
    broker = os.path.join(root, 'vvc_intra_b200/vvcb_broker')
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('LD_LIBRARY_PATH', None)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([broker, path, '--bit-depth', '10', '--clients', '8', '--frame', '128x128', '--workers', '3'], env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        procs = []
        for i, qp in enumerate((22, 27, 32, 37)):
            d = tmp_path / ('c%d' % i)
            d.mkdir()
            w, h = (128, 128) if i % 2 == 0 else (128, 64)
            Y, U, V = synth_yuv(w, h, 10, i)
            (d / 'in.yuv').write_bytes(Y.tobytes() + U.tobytes() + V.tobytes())
            (d / 'Time_python.dat').write_bytes(b'')
            procs.append((d, subprocess.Popen([plain] + _encoder_args(cfg, w, h, 10, qp) + ['-b', 'plain.bin'], cwd=d, env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True),
                          subprocess.Popen([served] + _encoder_args(cfg, w, h, 10, qp) + ['-b', 'gpu.bin'], cwd=d, env=dict(env0, VVCB_BROKER=path, VVCB_SHIM_REPORT=str(d / 'report.json')),
                                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for d, p1, p2 in procs:
            o1, _ = p1.communicate(timeout=900)
            o2, _ = p2.communicate(timeout=900)
            assert p1.returncode == 0, o1[-2000:]
            assert p2.returncode == 0, o2[-2000:]
            a, b = (d / 'plain.bin').read_bytes(), (d / 'gpu.bin').read_bytes()
            assert len(a) > 100 and a == b
        stats = json.loads(subprocess.check_output([broker, path, '--stats'], env=env0))
        print('broker stats', stats)
        assert stats['clients_seen'] == 4 and stats['max_batch'] >= 2 and stats['cycles'] < stats['requests'] and stats['kernel_launches'] > 1000
    finally:
        subprocess.run([broker, path, '--stop'], env=env0)
        try:
            out, _ = server.communicate(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
            out = ''
    assert server.returncode == 0, out[-2000:]


# ---- brief result records (vvcb_rmd_eval_brief) ------------------------------------------------------------------------
def _brief_matches(brief, full):
    from test_kernel_emulation import brief_matches
    return brief_matches(brief, full)


def test_brief_records_carry_the_same_lists(eng10):
    """vvcb_rmd_eval_brief (64-byte records) against vvcb_rmd_eval (368-byte records): counts, final list (whose first n_rd entries are the RD
    list) and Hadamard list, on random visits (one-shot path) and on a whole 1080p sweep (chunked copy / compute pipeline, trusted visits)."""
    rng = np.random.default_rng(141)
    orig, reco, visits = G.random_case(rng, 10, 12)
    eng10.frame_begin(orig)
    eng10.reco_update(reco)
    full = eng10.rmd_eval(visits)
    brief = eng10.rmd_eval_brief(visits)
    assert _brief_matches(brief, full)
    from bench import synth_luma, W, H
    frame = synth_luma(1)
    eng10.frame_begin(frame)
    eng10.reco_from_orig()                                  # == reco_update(frame), without the upload
    sweep = vb.build_sweep_visits(W, H, qp=27, ctu=128)
    assert len(sweep) > 600000
    eng10.set_option(vb.OPT_TRUSTED_VISITS, 1)
    try:
        b = eng10.rmd_eval_brief(sweep)
    finally:
        eng10.set_option(vb.OPT_TRUSTED_VISITS, 0)
    # the visits as a resident plan: same records
    d_plan = eng10.dev_alloc(sweep.nbytes)
    eng10.dev_upload(d_plan, sweep)
    b2 = eng10.rmd_eval_brief_resident(d_plan, len(sweep), np.zeros(len(sweep), vb.BRIEF_DTYPE))
    eng10.dev_free(d_plan)
    assert b2.tobytes() == b.tobytes()
    eng10.reco_update(frame)
    f = eng10.rmd_eval(sweep)
    assert np.array_equal(b['n_rd'], f['n_rd'].astype(np.uint8)) and np.array_equal(b['n_final'], f['n_final'].astype(np.uint8)) and np.array_equal(b['n_had'], f['n_had'].astype(np.uint8))
    code = f['final_mode']['mode'].astype(np.uint16) | (f['final_mode']['mrl'].astype(np.uint16) << 8) | (f['final_mode']['mip'].astype(np.uint16) << 15)
    mask = np.arange(16)[None, :] < f['n_final'][:, None]
    assert np.array_equal(np.where(mask, b['final_mode'], 0), np.where(mask, code, 0)) and not np.where(mask, 0, b['final_mode']).any()
    sel = rng.choice(len(sweep), 2000, replace=False)
    assert _brief_matches(b[sel], f[sel])
    bad = visits.copy()
    bad['log2w'][3] = 9
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.rmd_eval_brief(bad)


# ---- BASELINE.json configurations through the drop-in ------------------------------------------------------------------
def _run_served_vs_plain(tmp_path, cases, bits, frame_wh, workers=4):
    """cases: list of (name, Y, U, V, w, h, qp).  Plain and served encoders of all cases run concurrently (served ones share one broker);
    returns the broker statistics after checking bitstream AND reconstruction identity of every case."""
    import json
    import os
    import subprocess
    root, (plain, served, cfg) = _ref_binaries('EncoderApp', 'EncoderAppServe')
    broker = os.path.join(root, 'vvc_intra_b200/vvcb_broker')
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('LD_LIBRARY_PATH', None)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([broker, path, '--bit-depth', str(bits), '--clients', str(max(2, len(cases))), '--frame', '%dx%d' % frame_wh, '--workers', str(workers)],
                              env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        procs = []
        for name, Y, U, V, w, h, qp in cases:
            d = tmp_path / name
            d.mkdir()
            (d / 'in.yuv').write_bytes(Y.tobytes() + U.tobytes() + V.tobytes())
            (d / 'Time_python.dat').write_bytes(b'')
            args = _encoder_args(cfg, w, h, bits, qp)
            procs.append((d, subprocess.Popen([plain] + args + ['-b', 'plain.bin', '-o', 'plain.yuv'], cwd=d, env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True),
                          subprocess.Popen([served] + args + ['-b', 'gpu.bin', '-o', 'gpu.yuv'], cwd=d, env=dict(env0, VVCB_BROKER=path, VVCB_SHIM_REPORT=str(d / 'report.json')),
                                           stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        for d, p1, p2 in procs:
            o1, _ = p1.communicate(timeout=1500)
            o2, _ = p2.communicate(timeout=1500)
            assert p1.returncode == 0, o1[-2000:]
            assert p2.returncode == 0, o2[-2000:]
            a, b = (d / 'plain.bin').read_bytes(), (d / 'gpu.bin').read_bytes()
            assert len(a) > 100 and a == b, d.name
            assert (d / 'plain.yuv').read_bytes() == (d / 'gpu.yuv').read_bytes(), d.name          # reconstruction (after the loop filters) as well
            rep = json.loads((d / 'report.json').read_text())
            assert rep['enabled'] == 1 and rep['demand_round_trips'] == 0 and rep['stale_context'] == 0 and rep['tu_residual_bits_reference'] == 0, rep
        stats = json.loads(subprocess.check_output([broker, path, '--stats'], env=env0))
    finally:
        subprocess.run([broker, path, '--stop'], env=env0)
        try:
            server.communicate(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
    return stats


def test_config1_416x240_full_frame_served_is_bit_identical(tmp_path):
    """BASELINE.json configs[0]: encoder_intra.cfg, synthetic 416x240 8-bit 4:2:0, 1 frame, QP 32 (SURVEY.md App. G input) -- the whole frame
    through the served drop-in: bitstream and reconstruction equal the plain reference encoder's."""
    from make_golden import synth_yuv
    Y, U, V = synth_yuv(416, 240, 8)
    stats = _run_served_vs_plain(tmp_path, [('c1', Y, U, V, 416, 240, 32)], 8, (416, 240), workers=2)
    print('C1 broker stats', stats)
    assert stats['visits'] > 50000 and stats['tu_jobs'] > 1000000


def test_config2_1080p10_ctu_row_at_four_qps_served_is_bit_identical(tmp_path):
    """BASELINE.json configs[1] (bounded): the first CTU row of a 1920x1080 10-bit synthetic frame (1920x128, 15 CTUs) at QP 22, 27, 32 and 37,
    four encoder processes behind one broker: bitstreams and reconstructions equal the plain reference encoder's."""
    from make_golden import synth_yuv
    Y, U, V = synth_yuv(1920, 1080, 10)
    row = (Y[:128], U[:64], V[:64])
    cases = [('qp%d' % qp, row[0], row[1], row[2], 1920, 128, qp) for qp in (22, 27, 32, 37)]
    stats = _run_served_vs_plain(tmp_path, cases, 10, (1920, 128), workers=4)
    print('1080p10 CTU row broker stats', stats)
    assert stats['clients_seen'] == 4 and stats['visits'] > 400000 and stats['max_batch'] >= 2


def test_training_set_dump_through_the_feature_kernel(eng10, tmp_path):
    """GET_TRAINING_SET (EL/CABACWriter.cpp:515-858) on the device: every node of a random final coding tree of a 416x240 picture, features from
    vvcb_features_eval, the four .dat files; records equal the oracle's features, labels the tree's splits."""
    from test_host_features import random_tree, cu_lookup
    from make_golden import synth_yuv
    from vvc_intra_b200 import training_set as T
    Y = synth_yuv(416, 240, 8)[0].astype(np.int16)
    nodes, leaves = random_tree(np.random.default_rng(12), 416, 240)
    get_cu = cu_lookup(leaves, 416, 240)
    eng10.frame_begin(Y)
    n = T.dump_training_set(eng10, nodes, get_cu, str(tmp_path))
    jobs, labels = T.training_jobs(nodes, get_cu)
    assert n == len(jobs) > 100
    data = np.fromfile(tmp_path / 'Data_Partition.dat', '<i4').reshape(-1, 26)
    assert np.array_equal(data, O.features_batch(Y, jobs)['f'][:, :26])
    assert np.array_equal(np.fromfile(tmp_path / 'Label_Partition.dat', '<i4'), labels)


def test_cu_eval_templates_expand_over_the_lists(eng10):
    """vvcb_cu_auto: templates combined by the engine with the modes of the lists the same call produced (final list; regular-only list for the
    templates that ask for it; MIP modes dropped where told), in list order; every expanded candidate equals the same candidate submitted explicitly."""
    rng = np.random.default_rng(151)
    orig, reco, visits = G.random_case(rng, 10, 2, plane=(256, 512))
    eng10.frame_begin(orig)
    eng10.reco_update(reco)
    rates, states = vb.default_dq_rates(), vb.default_ctx_states()
    reqs = []
    for v in visits[:24]:
        au = np.zeros(3, vb.CU_AUTO_DTYPE)
        for k, (mts, lf, modes, skip) in enumerate(((0, 0, vb.AUTO_FINAL, 0), (2 if max(int(v['log2w']), int(v['log2h'])) <= 5 else 0, 0, vb.AUTO_FINAL | vb.AUTO_REGULAR, 0), (0, 1, vb.AUTO_REGULAR, 1))):
            j = au[k]['job']
            j['x'], j['y'], j['log2w'], j['log2h'], j['mts_idx'], j['lfnst_idx'] = v['x'], v['y'], v['log2w'], v['log2h'], mts, lf
            j['flags'] = vb.TU_QUANT | vb.TU_DEPQUANT | vb.TU_RATE
            j['qp_per'], j['qp_rem'], j['lambda'], j['cbf_delta_bits'] = 6, 3, 45.0, -1200
            au[k]['modes'], au[k]['skip_mip'] = modes, skip
        reqs.append(dict(visit=np.array([v]), want_rmd=True, autos=au, max_auto=64, rates=rates, states=states))
    outs = eng10.cu_eval(reqs)
    total = 0
    for q, o in zip(reqs, outs):
        v, res, det, au = q['visit'][0], o['result'][0], o['detail'][0], q['autos']
        n = int(o['n_auto'][0])
        final = [(int(m['mip']), int(m['mrl']), int(m['mode'])) for m in res['final_mode'][:res['n_final']]]
        reg = [(int(m['mip']), int(m['mrl']), int(m['mode'])) for m in det['reg_mode'][:det['n_reg']]]
        exp = []
        for (mip, mrl, mode), in_final in [(m, True) for m in final] + [(m, False) for m in reg if m not in final]:
            slot = vb.SLOT_MIP + mode if mip else mode if mrl == 0 else (vb.SLOT_MRL1 if mrl == 1 else vb.SLOT_MRL3) + list(v['mpm'][1:]).index(mode)
            for t in range(3):
                if (int(au[t]['modes']) & (vb.AUTO_FINAL if in_final else vb.AUTO_REGULAR)) and not (mip and au[t]['skip_mip']):
                    exp.append((slot, t))
        assert [(int(a), int(b)) for a, b in zip(o['auto_slot'][:n], o['auto_tmpl'][:n])] == exp[:64]
        # the same candidates submitted explicitly
        bs = 1 << (int(v['log2w']) + int(v['log2h']))
        jobs = np.zeros(n, vb.TU_JOB_DTYPE)
        for k in range(n):
            jobs[k] = au[int(o['auto_tmpl'][k])]['job']
            slot = int(o['auto_slot'][k])
            mode = 0 if slot >= vb.SLOT_MIP else slot if slot < vb.SLOT_MRL1 else int(v['mpm'][1 + (slot - vb.SLOT_MRL1) % 5])
            jobs[k]['offset'], jobs[k]['intra_mode'] = k * bs, mode if jobs[k]['lfnst_idx'] else 0
        o2 = eng10.cu_eval([dict(visit=q['visit'], jobs=jobs, slots=o['auto_slot'][:n].copy(), rates=rates, states=states)])[0]
        assert np.array_equal(o2['level'], o['auto_level'][:n * bs]) and np.array_equal(o2['reco'], o['auto_reco'][:n * bs]) and np.array_equal(o2['pred'], o['auto_pred'][:n * bs])
        assert o2['tu_results'].tobytes() == o['auto_results'][:n].tobytes()
        total += n
    assert total > 200
    bad = dict(reqs[0])
    bad['want_rmd'] = False
    with pytest.raises(vb.EngineError, match='malformed'):
        eng10.cu_eval([bad])


def test_frame_parallel_served_encode_gathers_to_the_sequential_bitstream(tmp_path):
    """The whole frame-parallel route (SURVEY.md 8e / 8f-4) on the GPU: one served encoder process per picture of a three-picture 10-bit sequence,
    all sharing one engine context through the broker; the gather (vvc_intra_b200/assemble.py) must reproduce the bitstream the plain sequential
    encoder writes for the sequence, byte for byte."""
    import json
    import os
    import subprocess
    from make_golden import synth_yuv
    from vvc_intra_b200 import assemble
    root, (plain, served, cfg) = _ref_binaries('EncoderApp', 'EncoderAppServe')
    broker = os.path.join(root, 'vvc_intra_b200/vvcb_broker')
    w, h, bits, qp, n = 128, 64, 10, 32, 3
    data = b''
    for f in range(n):
        Y, U, V = synth_yuv(w, h, bits, f)
        data += Y.tobytes() + U.tobytes() + V.tobytes()
    (tmp_path / 'in.yuv').write_bytes(data)
    (tmp_path / 'Time_python.dat').write_bytes(b'')
    args = _encoder_args(cfg, w, h, bits, qp)
    args = args[:args.index('-f')] + args[args.index('-f') + 2:]
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('LD_LIBRARY_PATH', None)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([broker, path, '--bit-depth', '10', '--clients', '4', '--frame', '128x64', '--workers', '2'], env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        seq = subprocess.Popen([plain] + args + ['-f', str(n), '-b', 'seq.bin'], cwd=tmp_path, env=env0, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        procs = [subprocess.Popen([served] + args + ['-f', '1', '--FrameSkip=%d' % f, '-b', 'f%d.bin' % f], cwd=tmp_path,
                                  env=dict(env0, VVCB_BROKER=path, VVCB_SHIM_REPORT=str(tmp_path / ('rep%d.json' % f))), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
                 for f in range(n)]
        for p in procs:
            out, _ = p.communicate(timeout=900)
            assert p.returncode == 0, out[-2000:]
        assert seq.wait(timeout=900) == 0
        stats = json.loads(subprocess.check_output([broker, path, '--stats'], env=env0))
        assert stats['clients_seen'] == n and stats['kernel_launches'] > 1000
    finally:
        subprocess.run([broker, path, '--stop'], env=env0)
        try:
            out, _ = server.communicate(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
            out = ''
    assert server.returncode == 0, out[-2000:]
    for f in range(n):
        assert json.loads((tmp_path / ('rep%d.json' % f)).read_text())['visits'] > 100
    stats = assemble.assemble_sequential([str(tmp_path / ('f%d.bin' % f)) for f in range(n)], str(tmp_path / 'all.bin'))
    assert (tmp_path / 'all.bin').read_bytes() == (tmp_path / 'seq.bin').read_bytes()
    print('frame-parallel gather', stats)
