"""One context serving every entry point in turn.

A context keeps its scratch memory in grow-only slots (vvcb_api.cu): a slot that is too small is freed and allocated anew, and a larger
one keeps serving smaller calls.  vvcb_cu_eval's first stage, vvcb_isp_eval and vvcb_chroma_tu_eval share the staging slots.  Here one
context runs vvcb_cu_eval (walk), vvcb_tu_eval_pred, vvcb_isp_eval, vvcb_chroma_eval, vvcb_chroma_tu_eval, vvcb_features_eval and
vvcb_rmd_eval_brief in turn, at batch sizes that grow and then shrink, so that every slot these calls use is reallocated and the shared
ones pass from one entry point to the next.  Each call's outputs must equal, byte for byte, those of the same call on a fresh context.

Also: the functions that a context reached through the broker proxy does not serve refuse with VVCB_ERR_STATE."""
import os
import subprocess
import sys
import time

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BD, W, H = 10, 512, 256
SCALES = (1, 6, 30, 6, 1)                     # batch size factor of each round: the slots grow twice, then serve smaller calls
QUANT, DEPQUANT, RATE = 1, 2, 32
# luma CU shapes (log2): those of the sweep planner (vvc_intra_b200.partition), sides 4..32 and 64x64.  A 64-sample side with an aspect
# ratio of 4 or more is left out: on reference lines 1 / 3 its replicated tail exceeds the kLineMax line arrays of the RMD kernels.
SHAPES = [(lw, lh) for lw in range(2, 6) for lh in range(2, 6)] + [(6, 6)]


def E():
    import vvc_intra_b200.engine as eng
    return eng


def planes():
    rng = np.random.default_rng(17)
    luma, reco = (rng.integers(0, 1 << BD, (H, W)).astype(np.int16) for _ in range(2))
    cb, cr, cb_reco, cr_reco = (rng.integers(0, 1 << BD, (H // 2, W // 2)).astype(np.int16) for _ in range(4))
    return luma, reco, cb, cr, cb_reco, cr_reco


def prepared(p):
    import vvc_intra_b200 as vb
    luma, reco, cb, cr, cb_reco, cr_reco = p
    eng = vb.IntraCostEngine(device=0, bit_depth=BD, ctu_size=128)
    eng.frame_begin(luma)
    eng.reco_update(reco)
    eng.chroma_frame_begin(cb, cr)
    eng.chroma_reco_update(cb_reco, cr_reco)
    return eng


def luma_visits(rng, n):
    """n visits of random shapes (SHAPES) with full left / above availability inside the picture"""
    v = np.zeros(n, E().VISIT_DTYPE)
    lw, lh = np.array(SHAPES)[rng.integers(0, len(SHAPES), n)].T
    w, h = 1 << lw, 1 << lh
    v['log2w'], v['log2h'] = lw, lh
    v['x'] = 4 * rng.integers(1, (W - 2 * w) // 4 + 1)
    v['y'] = 4 * rng.integers(1, (H - 2 * h) // 4 + 1)
    v['avail_al'], v['n_above'], v['n_above_right'], v['n_left'], v['n_below_left'] = 1, w // 4, w // 4, h // 4, h // 4
    v['mpm'] = [0, 50, 18, 46, 54, 1]
    v['num_mpm_cand'] = 3
    v['rates'] = rng.integers(1000, 90000, (n, v['rates'].shape[1]))
    v['sqrt_lambda'] = 0.002
    return v


def tu_jobs(visits, per_visit, rng):
    """per_visit dependent-quantisation TU jobs (regular modes) on the geometry of each visit; returns (jobs, slots, n_samples)"""
    vb = E()
    idx = np.repeat(np.arange(len(visits)), per_visit)
    j = np.zeros(len(idx), vb.TU_JOB_DTYPE)
    for k in ('x', 'y', 'log2w', 'log2h'):
        j[k] = visits[k][idx]
    j['flags'] = vb.TU_QUANT | vb.TU_DEPQUANT | vb.TU_RATE
    qp = rng.integers(22, 42, len(j))
    j['qp_per'], j['qp_rem'] = qp // 6, qp % 6
    j['lambda'] = 0.57 * 2.0 ** ((qp - 12) / 3.0) * 16
    sizes = 1 << (j['log2w'].astype(np.int64) + j['log2h'].astype(np.int64))
    j['offset'] = np.concatenate(([0], np.cumsum(sizes)[:-1]))
    return j, rng.integers(0, 67, len(j)).astype(np.uint8), int(sizes.sum())


def call_cu_eval(rng, s):
    import vvc_intra_b200 as vb
    visits = luma_visits(rng, s)
    reqs = []
    for i in range(s):
        v = visits[i:i + 1]
        jobs, slots, _ = tu_jobs(v, 6, rng)
        reqs.append(dict(visit=v, want_rmd=1, jobs=jobs, slots=slots, rates=vb.default_dq_rates(), states=vb.default_ctx_states()))
    return lambda eng: [a for o in eng.cu_eval(reqs) for a in o.values()]


def call_tu_eval_pred(rng, s):
    import vvc_intra_b200 as vb
    visits = luma_visits(rng, 2 * s)
    jobs, slots, ns = tu_jobs(visits, 3, rng)
    src = np.zeros(len(jobs), vb.TU_SRC_DTYPE)
    src['visit'], src['slot'] = np.repeat(np.arange(len(visits)), 3), slots
    return lambda eng: list(eng.tu_eval_pred(visits, src, jobs, ns, want_coeff=True, want_level=True, want_reco=True, want_pred=True,
                                             rates=vb.default_dq_rates(), states=vb.default_ctx_states()).values())


def call_isp_eval(rng, s):
    from isp_eval_probe import HOR, VER, blocks, job, states
    visits = luma_visits(rng, 2 * s)
    visits['n_below_left'] = 0
    jobs, off = [], 0
    for c, v in enumerate(visits):
        w, h = 1 << int(v['log2w']), 1 << int(v['log2h'])
        for isp in (HOR, VER):
            if w * h > 16 and min(blocks(w, h, isp == HOR)) >= 4:
                for mode in rng.choice(67, 2, replace=False):
                    jobs.append(job(len(jobs), c, isp, int(mode), int(rng.integers(22, 42)), off))
                    off += w * h
    jobs = np.array(jobs, E().ISP_JOB_DTYPE)
    st = states(rng, len(jobs))
    return lambda eng: list(eng.isp_eval(visits, jobs, off, states=st, want_level=True, want_reco=True, want_pred=True).values())


def chroma_visits(rng, n):
    from chroma_eval_probe import sweep_visits
    sweep = sweep_visits(rng, W // 2, H // 2)
    return sweep[rng.choice(len(sweep), n, replace=False)]


def call_chroma_eval(rng, s):
    visits = chroma_visits(rng, 4 * s)
    return lambda eng: (lambda r: [r[0]] + r[1])(eng.chroma_eval(visits, want_pred=True))


def call_chroma_tu_eval(rng, s):
    from chroma_tu_probe import jobs_for, states
    visits = chroma_visits(rng, 3 * s)
    jobs, ns = jobs_for(visits, 3, rng, qp=int(rng.integers(22, 42)))
    st = states(rng, 1)
    return lambda eng: list(eng.chroma_tu_eval(visits, jobs, ns, states=st, want_level=True, want_reco=True, want_pred=True).values())


def call_features_eval(rng, s):
    from test_oracle_features import random_feature_jobs
    jobs = random_feature_jobs(rng, H, W, 40 * s)
    return lambda eng: [eng.features_eval(jobs)]


def call_rmd_eval_brief(rng, s):
    visits = luma_visits(rng, 30 * s)
    return lambda eng: [eng.rmd_eval_brief(visits)]


CALLS = (call_cu_eval, call_tu_eval_pred, call_isp_eval, call_chroma_eval, call_chroma_tu_eval, call_features_eval, call_rmd_eval_brief)


@pytest.mark.gpu
def test_interleaved_entry_points_equal_fresh_contexts():
    p = planes()
    rng = np.random.default_rng(23)
    shared = prepared(p)
    try:
        for r, s in enumerate(SCALES):
            for make in CALLS:
                run = make(rng, s)
                got = run(shared)
                fresh = prepared(p)
                try:
                    exp = run(fresh)
                finally:
                    fresh.close()
                name = '%s (round %d, scale %d)' % (make.__name__[5:], r, s)
                assert len(got) == len(exp), name
                for k, (a, b) in enumerate(zip(got, exp)):
                    assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), (name, k)
    finally:
        shared.close()


@pytest.mark.gpu
def test_broker_proxy_refuses_local_memory_and_timer(tmp_path):
    """vvcb_dev_alloc, vvcb_host_alloc and vvcb_timer_stop act on the local device: a context reached through the broker proxy
    refuses them with VVCB_ERR_STATE, as it refuses vvcb_dev_free, vvcb_host_free and vvcb_timer_start."""
    path = str(tmp_path / 'broker.shm')
    env0 = dict(os.environ)
    env0.pop('VVCB_BROKER', None)
    server = subprocess.Popen([os.path.join(ROOT, 'vvc_intra_b200/vvcb_broker'), path, '--bit-depth', '10', '--ctu', '128', '--clients', '2',
                               '--frame', '320x256', '--workers', '1'], env=env0, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        prog = ('import ctypes as C, vvc_intra_b200 as vb\n'
                'eng = vb.IntraCostEngine(device=0, bit_depth=10, ctu_size=128)\n'
                'L, ctx, p, ms = eng._lib, eng._ctx, C.c_void_p(), C.c_float()\n'
                'for name, call in (("vvcb_dev_alloc", lambda: L.vvcb_dev_alloc(ctx, 64, C.byref(p))),\n'
                '                   ("vvcb_host_alloc", lambda: L.vvcb_host_alloc(ctx, 64, C.byref(p))),\n'
                '                   ("vvcb_timer_stop", lambda: L.vvcb_timer_stop(ctx, C.byref(ms)))):\n'
                '    rc = call()\n'
                '    print(name, rc, L.vvcb_last_error(ctx).decode() == name + ": not available through the broker")\n')
        r = None
        for _ in range(100):
            if os.path.exists(path):
                r = subprocess.run([sys.executable, '-c', prog], cwd=ROOT, env=dict(env0, VVCB_BROKER=path), stdout=subprocess.PIPE,
                                   stderr=subprocess.STDOUT, text=True, timeout=300)
                break
            time.sleep(0.2)
        assert r is not None and r.returncode == 0, r and r.stdout[-2000:]
        assert r.stdout.strip().splitlines()[-3:] == ['vvcb_dev_alloc -3 True', 'vvcb_host_alloc -3 True', 'vvcb_timer_stop -3 True'], r.stdout[-2000:]
    finally:
        subprocess.run([os.path.join(ROOT, 'vvc_intra_b200/vvcb_broker'), path, '--stop'], env=env0, timeout=60)
        try:
            server.wait(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
