#!/usr/bin/env python
"""bench.py -- throughput of the intra cost-evaluation hot path (BASELINE.json: all-intra 1080p10 CTUs/sec).

b200 arm (default): one "step" = the exhaustive rough-mode-decision sweep of ONE 1920x1080 10-bit frame:
every candidate luma CU of every 64x64 root (679 260 visits, SURVEY.md App. C) x every evaluation slot
(67 regular modes, MPMs on reference lines 1 and 3, all MIP modes): reference-line fetch, prediction,
SAD, SATD, mode bits, costs and the reference's candidate lists.  Steps cycle over 8 synthetic frames
and QP 32/27/37/22.  `value` times the kernels with planes, visits and results resident in HBM; `e2e`
times the same step through the C ABI with HOST buffers (page-locked), copies included.

reference arm (--impl reference): the UNMODIFIED reference encoder (oracle/_ref/EncoderApp, built by
__graft_entry__.build() from /root/reference) on the box's host cores, one process per 128x128 crop of
the same synthetic frames -- a bounded sample of the same workload, all cores busy.

Launch: python bench.py --gpus N --steps K --warmup W   (N > 1 under torchrun, one rank per GPU).
--dump-outputs DIR writes the result records of the last timed step as .npy files, to compare two builds output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, 'tools')):
    if p not in sys.path:
        sys.path.insert(0, p)

W, H, BITS, NFRAMES = 1920, 1080, 10, 8
QPS = (32, 27, 37, 22)
CTU = 128
CTUS_PER_FRAME = ((W + CTU - 1) // CTU) * ((H + CTU - 1) // CTU)     # 15 x 9 = 135


def synth_luma(frame):
    from make_golden import synth_yuv
    return synth_yuv(W, H, BITS, frame)[0].astype(np.int16)


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe): NVML polled every few milliseconds from a
    thread of this process (the timed region of the default run is ~150 ms, too short for `nvidia-smi -lms`); nvidia-smi as a fallback."""
    REASONS = (('hw_slowdown', 0x8), ('hw_thermal_slowdown', 0x40), ('sw_thermal_slowdown', 0x20), ('sw_power_cap', 0x4))

    def __init__(self, index):
        self.index, self.rows, self.stop, self.thread, self.smi = index, [], threading.Event(), None, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def _poll(self):
        nv = self.nv
        while not self.stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                self.rows.append((sm, self.max_sm, mask))
            except Exception:
                pass
            self.stop.wait(0.004)

    def _read_smi(self):
        for line in self.smi.stdout:
            c = [x.strip() for x in line.split(',')]
            try:
                mask = sum(bit for (_, bit), v in zip(self.REASONS, c[2:6]) if v.lower().startswith('active'))
                self.rows.append((float(c[0]), float(c[1]), mask))
            except (ValueError, IndexError):
                continue

    def __enter__(self):
        if self.nv is not None:
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
        else:
            try:
                q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
                     'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
                self.smi = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '20'],
                                            stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                self.thread = threading.Thread(target=self._read_smi, daemon=True)
                self.thread.start()
            except OSError:
                self.smi = None
        return self

    def __exit__(self, *a):
        self.stop.set()
        if self.smi:
            time.sleep(0.05)
            self.smi.terminate()
        if self.thread:
            self.thread.join(timeout=2)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return {'sm_mhz': statistics.median(r[0] for r in self.rows), 'sm_max_mhz': max(r[1] for r in self.rows),
                'reasons': sorted(name for name, bit in self.REASONS if mask & bit), 'samples': len(self.rows),
                'source': 'nvml' if self.nv is not None else 'nvidia-smi'}


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))), 'measured (MEASURED_PEAKS.json)'
    except OSError:
        return {'hbm_gbs': 6650.0}, 'fallback (B200_PROFILING.md)'


def eval_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the rmd_eval_kernel launches (33: per tile class and prediction kind, packed small shapes and larger shapes) of one 1080p step, from the committed
    ncu capture (profiles/eval_traffic.json, written by tools/make_traffic.py on the GPU box)."""
    try:
        t = json.load(open(os.path.join(ROOT, 'profiles', 'eval_traffic.json')))
        return t['dram_bytes_per_step'], t['source']
    except (OSError, KeyError, ValueError):
        return None, None


def active_slot_counts(vis):
    """Evaluation slots per visit, as the kernels count them."""
    w, h = 1 << vis['log2w'].astype(np.int64), 1 << vis['log2h'].astype(np.int64)
    mip = np.where((w > 4 * h) | (h > 4 * w), 0, np.where((w == 4) & (h == 4), 35, np.where((w <= 8) & (h <= 8), 19, 11)))
    mrl = np.where((vis['y'].astype(np.int64) & (CTU - 1)) != 0, 10, 0)
    return 67 + mrl + mip, w * h


def run_b200(args, rank, world, local_rank, dist):
    import vvc_intra_b200 as vb
    peaks, peak_src = measured_peaks()
    eng = vb.IntraCostEngine(device=local_rank, bit_depth=BITS, ctu_size=CTU)
    base = vb.build_sweep_visits(W, H, qp=32, ctu=CTU)
    n = len(base)
    slots, area = active_slot_counts(base)
    evals_per_step = int(slots.sum())
    samples_per_step = int((slots * area).sum())
    # SURVEY.md 8d: algorithmic integer ops per predicted sample = 13 + log2(tile w) + log2(tile h)
    satd_ops = np.where((area == 16), 6, np.where(np.minimum(1 << base['log2w'].astype(int), 1 << base['log2h'].astype(int)) == 4, 7,
                        np.where(base['log2w'] == base['log2h'], 8, 9)))
    ops_per_step = float((slots * area * (13 + satd_ops)).sum())
    # algorithmic bytes per step: visit descriptors in, result lists out, SAD+SATD of every evaluation written and read once
    # (slot-major scratch), original samples once per visit, reference lines (2w+2h+1 samples per line, 3 lines)
    w_, h_ = 1 << base['log2w'].astype(np.int64), 1 << base['log2h'].astype(np.int64)
    bytes_per_step = float(n * (vb.VISIT_DTYPE.itemsize + vb.RESULT_DTYPE.itemsize) + 2 * 2 * 4 * evals_per_step
                           + (2 * area).sum() + (3 * 2 * (2 * w_ + 2 * h_ + 1)).sum())

    frames = [synth_luma(f) for f in range(NFRAMES)]
    # this rank's share of the (frame, qp) pairs: all-intra frames are independent -> no collective on the path
    mine = vb.shard.shard_units(vb.shard.work_units(NFRAMES, QPS), rank, world)

    # ---- resident set-up
    pitch = (W + 63) & ~63
    d_planes = []
    for f in range(NFRAMES):
        padded = np.zeros((H, pitch), np.int16)
        padded[:, :W] = frames[f]
        d = eng.dev_alloc(padded.nbytes)
        eng.dev_upload(d, padded)
        d_planes.append(d)
    d_vis = {}
    for qp in QPS:
        v = base.copy()
        v['sqrt_lambda'] = vb.partition.sqrt_lambda_for_qp(qp)
        d = eng.dev_alloc(v.nbytes)
        eng.dev_upload(d, v)
        d_vis[qp] = d
    d_res = eng.dev_alloc(n * vb.RESULT_DTYPE.itemsize)

    def resident_step(s):
        f, qp = mine[s % len(mine)]
        eng.frame_bind_device(d_planes[f], d_planes[f], pitch, W, H)     # speculative sweep: neighbours from the original
        eng.rmd_eval_device(d_vis[qp], n, d_res, None)       # detail tables are optional and not requested here

    int_peak = eng.measure_int_peak()
    for s in range(args.warmup):
        resident_step(s)
    eng.sync()
    if dist is not None:
        dist.barrier()
    eng.kernel_timing(True)
    launches0 = eng.launch_count
    with ClockSampler(local_rank) as clk:
        eng.sync()
        eng.timer_start()
        for s in range(args.steps):
            resident_step(args.warmup + s)
        ms_total = eng.timer_stop()
        eng.sync()
    k_plan, k_eval, k_lists, k_n = eng.kernel_times()
    eng.kernel_timing(False)
    launches = eng.launch_count - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, eng, vb, d_res, n)
    ms_total = vb.shard.max_over_ranks(ms_total, dist, 'cuda:%d' % local_rank)

    e2e_s, e2e_steps, e2e_full_s, e2e_plan_s = float("nan"), 1, float("nan"), float("nan")
    if not args.resident_only:
        # ---- end to end through the C ABI with host buffers
        h_vis = {}
        for qp in QPS:
            a = eng.host_array(n, vb.VISIT_DTYPE)
            a[:] = base
            a['sqrt_lambda'] = vb.partition.sqrt_lambda_for_qp(qp)
            h_vis[qp] = a
        h_res = eng.host_array(n, vb.BRIEF_DTYPE)
        h_frames = []
        for f in range(NFRAMES):
            a = eng.host_array(H * W, np.int16).reshape(H, W)
            a[:] = frames[f]
            h_frames.append(a)
        # the sweep's visits come from this process's own planner (vvc_intra_b200.partition): no host-side re-validation of 679 260 structs per step
        eng.set_option(vb.OPT_TRUSTED_VISITS, 1)

        def e2e_step(s):
            f, qp = mine[s % len(mine)]
            eng.frame_begin(h_frames[f])
            eng.reco_from_orig()                           # the sweep's neighbours are the original picture: copied on the device
            eng.rmd_eval_brief(h_vis[qp], out=h_res)       # 64-byte records: the mode lists the walk consumes
            return int(h_res['n_rd'][0])

        e2e_steps = max(1, args.steps)
        for s in range(2):
            e2e_step(s)
        eng.sync()
        if dist is not None:
            dist.barrier()
        t0 = time.perf_counter()
        for s in range(e2e_steps):
            e2e_step(2 + s)
        eng.sync()
        e2e_s = time.perf_counter() - t0
        e2e_s = vb.shard.max_over_ranks(e2e_s, dist, 'cuda:%d' % local_rank)
        eng.set_option(vb.OPT_TRUSTED_VISITS, 0)
        # the same step with the visit plan resident on the device (it is the same for every picture of a QP): only the picture goes up
        t0 = time.perf_counter()
        for s in range(4):
            f, qp = mine[s % len(mine)]
            eng.frame_begin(h_frames[f])
            eng.reco_from_orig()
            eng.rmd_eval_brief_resident(d_vis[qp], n, h_res)
        eng.sync()
        e2e_plan_s = (time.perf_counter() - t0) / 4
        # the same through the full 368-byte records (costs as doubles, three lists), for the record
        h_full = eng.host_array(n, vb.RESULT_DTYPE)
        eng.rmd_eval(h_vis[QPS[0]], out=h_full)
        eng.sync()
        t0 = time.perf_counter()
        for s in range(2):
            f, qp = mine[s % len(mine)]
            eng.frame_begin(h_frames[f])
            eng.reco_update(h_frames[f])
            eng.rmd_eval(h_vis[qp], out=h_full)
        eng.sync()
        e2e_full_s = (time.perf_counter() - t0) / 2
    h2d = H * W * 2 + n * vb.VISIT_DTYPE.itemsize
    d2h = n * vb.BRIEF_DTYPE.itemsize

    strong = None if (args.no_strong or args.resident_only) else strong_scaling_leg(eng, vb, rank, world, dist, local_rank)
    if rank != 0:
        return
    tu_stage = None if (args.no_tu_stage or args.resident_only) else tu_stage_leg(eng, vb, base, frames[0], int_peak)
    feat_stage = None if (args.no_tu_stage or args.resident_only) else features_stage_leg(eng, vb, frames[0])
    ms_step = ms_total / args.steps
    value = world * args.steps * CTUS_PER_FRAME / (ms_total * 1e-3)
    eval_ms = k_eval / max(1, k_n)
    hbm_achieved = bytes_per_step / (eval_ms * 1e-3) / 1e9 if eval_ms > 0 else 0.0
    int_best = max(int_peak)
    traffic, traffic_src = eval_traffic()
    out = {
        'metric': 'all-intra 1080p10 CTUs/sec (exhaustive RMD sweep: intra pred + SAD/SATD + mode cost + candidate lists)',
        'value': value, 'unit': 'CTU/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms_step, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'int16 samples / int32 arithmetic / f64 costs', 'data': 'synthetic',
        'config': {'workload': 'configs[1]: all-intra 1920x1080 10-bit synthetic YUV, 8 frames, QP 22/27/32/37, one frame sweep per step',
                   'visits_per_step': n, 'satd_evals_per_step': evals_per_step, 'ctus_per_step': CTUS_PER_FRAME,
                   'predicted_samples_per_step': samples_per_step,
                   'l2': 'per-step working set %.2f GB (visits + SAD/SATD scratch + result lists) > 126 MB L2; consecutive steps use different frames' %
                         ((n * (vb.VISIT_DTYPE.itemsize + vb.RESULT_DTYPE.itemsize + 2 * 4 * 112)) / 1e9),
                   'sharding': 'frames x QPs partitioned across ranks, no collective on the hot path'},
        'satd_evals_per_s': world * args.steps * evals_per_step / (ms_total * 1e-3),
        'e2e': {'value': world * e2e_steps * CTUS_PER_FRAME / e2e_s, 'unit': 'CTU/s', 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'steps': e2e_steps,
                'resident_plan_ctus_per_s': world * CTUS_PER_FRAME / e2e_plan_s, 'resident_plan_h2d_bytes_per_step': H * W * 2,
                'full_records_ctus_per_s': world * CTUS_PER_FRAME / e2e_full_s, 'full_records_d2h_bytes_per_step': n * vb.RESULT_DTYPE.itemsize,
                'note': 'vvcb_frame_begin + vvcb_reco_from_orig + vvcb_rmd_eval_brief (64-byte records: the mode lists) with page-locked host buffers, wall clock; '
                        'resident_plan_*: the visits (a static plan, identical for every picture of a QP) stay on the device, vvcb_rmd_eval_brief_resident; '
                        'full_records_*: the same step through vvcb_rmd_eval (368-byte records with the double costs)'},
        'gpu_launches': launches,
        'clocks': clk.summary(),
        # the dominant kernels are integer-issue bound (SURVEY.md 8d): the roofline is the measured integer issue peak; the HBM view is kept beside it
        'roofline': {'bound': 'int_alu', 'kernel': 'rmd_eval_kernel', 'achieved': ops_per_step / (eval_ms * 1e-3) / 1e12 if eval_ms > 0 else 0.0,
                     'peak': int_best / 1e3, 'unit': 'Tera lane-ops/s', 'frac': (ops_per_step / (eval_ms * 1e-3) / 1e9) / int_best if eval_ms > 0 and int_best else None,
                     'traffic': traffic, 'traffic_source': traffic_src,
                     'peak_source': 'measured live (vvcb_measure_int_peak): dependent-free IMAD / IADD3+LOP3 / mixed streams = %.0f / %.0f / %.0f Gop/s; MEASURED_PEAKS.json has no integer peak' % int_peak,
                     'kernel_ms': eval_ms, 'kernel_share_of_step': eval_ms / ms_step if ms_step else None,
                     'algorithmic_ops_per_launch': ops_per_step,
                     'ops_model': 'SURVEY.md 8d: 13 + (6|7|8|9 by SATD tile) = 19..22 integer ops per predicted sample',
                     'hbm': {'achieved_gbs': hbm_achieved, 'peak_gbs': peaks.get('hbm_gbs'), 'frac': hbm_achieved / peaks.get('hbm_gbs') if peaks.get('hbm_gbs') else None,
                             'algorithmic_bytes_per_launch': bytes_per_step, 'peak_source': peak_src}},
        'int_alu': {'achieved_gops': ops_per_step / (eval_ms * 1e-3) / 1e9 if eval_ms > 0 else 0.0,
                    'peak_gops': int_best, 'frac': (ops_per_step / (eval_ms * 1e-3) / 1e9) / int_best if eval_ms > 0 and int_best else None},
        'kernel_ms': {'plan': k_plan / max(1, k_n), 'eval': eval_ms, 'lists': k_lists / max(1, k_n)},
    }
    if strong:
        out['strong_scaling'] = strong
    if tu_stage:
        out['tu_stage'] = tu_stage
    if feat_stage:
        out['features_stage'] = feat_stage
    if world == 1 and not args.no_cpu_baseline and not args.resident_only:
        out['cpu_baseline'] = cpu_baseline_port(base, frames[0])
    if world == 1 and not args.no_bitexact and not args.resident_only:
        out['bitexact'] = bitexact_leg(frames, local_rank)
    emit(out)


DUMP_VISITS = 1 << 16      # 46 MB of arrays; all 679 260 records would be 250 MB


def dump_outputs(out_dir, eng, vb, d_res, n):
    """--dump-outputs: the result records of the last timed step, as vvcb_rmd_eval_device hands them to its caller, for a fixed
    seeded sample of the step's visits.  One float array per field: list lengths (n_rd, n_had, n_final), costs, and the
    (mip, mrl, mode) triple of every list entry; entries past a list's length are zero, as the kernel writes them."""
    res = np.empty(n, vb.RESULT_DTYPE)
    eng.dev_download(res, d_res)
    idx = np.sort(np.random.default_rng(7).choice(n, min(n, DUMP_VISITS), replace=False))
    r = res[idx]
    arrays = {'visit_index': idx.astype(np.float64),
              'list_lengths': np.stack([r['n_rd'], r['n_had'], r['n_final']], axis=1).astype(np.float64),
              'rd_cost': r['rd_cost'].astype(np.float64), 'had_cost': r['had_cost'].astype(np.float64)}
    for f in ('rd_mode', 'had_mode', 'final_mode'):
        arrays[f] = np.stack([r[f]['mip'], r[f]['mrl'], r[f]['mode']], axis=-1).astype(np.float32)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def strong_scaling_leg(eng, vb, rank, world, dist, local_rank):
    """BASELINE.json configs[2]: 64 frames of 3840x2160 10-bit, a FIXED job sharded by frame over the ranks (frame f -> rank f mod N), through the
    host-buffer entry points (planes and visits up, brief records down), ending with the gather of the per-frame statistics on every rank.
    Wall clock around the whole job, max over ranks; the driver's SCALE run gives it at N = 1, 2, 4, 8."""
    from make_golden import synth_yuv
    w4, h4, n_frames, qp = 3840, 2160, 64, 32
    vis = vb.build_sweep_visits(w4, h4, qp=qp, ctu=CTU)
    n = len(vis)
    d_plan = eng.dev_alloc(vis.nbytes)                # the sweep's visits are a static plan: uploaded once per rank, outside the job
    eng.dev_upload(d_plan, vis)
    hr = eng.host_array(n, vb.BRIEF_DTYPE)
    # four distinct synthetic 2160p frames (generating 64 takes longer than encoding them); frame f of the job is picture f % 4
    pics = []
    for f in range(4):
        a = eng.host_array(h4 * w4, np.int16).reshape(h4, w4)
        a[:] = synth_yuv(w4, h4, BITS, f)[0]
        pics.append(a)
    mine = [f for f in range(n_frames) if f % world == rank]
    eng.frame_begin(pics[0]); eng.reco_from_orig(); eng.rmd_eval_brief_resident(d_plan, n, hr)      # warm-up: allocations, pipeline buffers
    eng.sync()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    stats = []
    for f in mine:
        eng.frame_begin(pics[f % 4])
        eng.reco_from_orig()
        eng.rmd_eval_brief_resident(d_plan, n, hr)
        sample = hr[::16]                                   # per-frame statistics of the chosen lists (every 16th visit: the host pass stays off the critical path)
        stats.append((f, int(sample['n_final'].sum()), int(sample['final_mode'][:, 0].astype(np.int64).sum())))
    eng.sync()
    merged = vb.shard.gather_stats(stats, dist)
    dt = vb.shard.max_over_ranks(time.perf_counter() - t0, dist, 'cuda:%d' % local_rank)
    eng.dev_free(d_plan)
    if sorted(m[0] for m in merged) != list(range(n_frames)):
        raise SystemExit('bench: the strong-scaling gather lost frames')
    ctus = ((w4 + CTU - 1) // CTU) * ((h4 + CTU - 1) // CTU)
    return {'workload': 'configs[2]: 64 frames 3840x2160 10-bit, exhaustive RMD sweep (%d visits per frame), sharded by frame over %d rank(s); per frame the picture goes up and the brief records come down (host buffers), the visit plan is resident; final statistics gather' % (n, world),
            'scaling': 'strong', 'n_gpus': world, 'seconds': dt, 'frames_per_s': n_frames / dt, 'ctus_per_s': n_frames * ctus / dt,
            'h2d_bytes_per_frame': int(h4 * w4 * 2), 'd2h_bytes_per_frame': int(n * vb.BRIEF_DTYPE.itemsize),
            'stats_checksum': int(sum(m[1] + m[2] for m in merged) & 0xffffffff)}


def features_stage_leg(eng, vb, frame):
    """configs[3]: the FAST_ALGORITHM classifier inputs (EL/EncCu.cpp:816-1138) of every candidate CU of a 1080p 10-bit frame (4x4
    excluded as in the reference) plus the per-CTU Hadamard texture sums (EncCu::updateCtuDataISlice), through the host-buffer
    entry points (job upload and result download inside the timed region); its own unit (CUs/s), next to the oracle on one core."""
    from oracle import oracle_py as O
    from vvc_intra_b200.features import build_sweep_feature_jobs
    eng.frame_begin(frame)
    jobs = build_sweep_feature_jobs(W, H)
    hj = eng.host_array(len(jobs), vb.FEAT_JOB_DTYPE)
    hj[:] = jobs
    eng.features_eval(hj[:4096])
    eng.sync()
    t0 = time.perf_counter()
    reps = 3
    for _ in range(reps):
        res = eng.features_eval(hj)
        had = eng.ctu_hads_islice(W, H)
    wall = (time.perf_counter() - t0) / reps
    sample = jobs[::5]
    t0 = time.perf_counter()
    exp = O.features_batch(frame, sample)
    cpu_s = time.perf_counter() - t0
    if exp.tobytes() != res[::5].tobytes() or had.tolist() != O.ctu_hads_islice(frame, ctu=CTU).tolist():
        raise SystemExit('bench: features differ from the oracle')
    return {'workload': 'configs[3]: 27 classifier features of the %d candidate CUs of frame 0 (1920x1080 10-bit; the picture-size gate of the '
                        'reference, hard-coded 416x240, not applied) + per-CTU Hadamard sums' % len(jobs),
            'cus_per_s_e2e': len(jobs) / wall, 'e2e_ms': wall * 1e3, 'h2d_bytes': int(jobs.nbytes), 'd2h_bytes': int(res.nbytes + had.nbytes),
            'valid_fraction': float((res['valid'] != 0).mean()),
            'cpu_baseline': {'value': len(sample) / cpu_s, 'unit': 'CU/s', 'cores': 1, 'kind': 'port',
                             'sample': 'oracle/vvc_oracle_feat.c on every 5th job (%d jobs, %.1f s); the same jobs are compared bit-exactly' % (len(sample), cpu_s)}}


def tu_stage_leg(eng, vb, base, frame, int_peak):
    """Second stage of the cost evaluation, reported next to the headline (its own unit: TUs/s): for every candidate CU of frame 0
    the best candidate of its rough-mode-decision list goes through vvcb_tu_eval_pred -- intra prediction, residual, forward
    DCT-II, dependent quantisation, inverse, reconstruction, SSE (IntraSearch::xIntraCodingTUBlock) -- with host buffers for the
    job descriptions and results; kernel times from CUDA events around each launch."""
    from oracle import oracle_py as O
    eng.frame_begin(frame)
    eng.reco_update(frame)
    vis = base.copy()
    vis['sqrt_lambda'] = vb.partition.sqrt_lambda_for_qp(32)
    res = eng.rmd_eval(vis)
    src, jobs, n_samples, rates = vb.build_tu_jobs_from_lists(vis, res, 32, BITS, rate=True)
    states = vb.default_ctx_states()
    hv = eng.host_array(len(vis), vb.VISIT_DTYPE)
    hv[:] = vis
    hs = eng.host_array(len(src), vb.TU_SRC_DTYPE)
    hs[:] = src
    hj = eng.host_array(len(jobs), vb.TU_JOB_DTYPE)
    hj[:] = jobs
    eng.tu_eval_pred(hv, hs, hj, n_samples, rates=rates, states=states)      # warm-up (allocations)
    eng.kernel_timing(True)
    reps = 3
    t0 = time.perf_counter()
    for _ in range(reps):
        out = eng.tu_eval_pred(hv, hs, hj, n_samples, rates=rates, states=states)
    wall = (time.perf_counter() - t0) / reps
    k_tr, k_dq, k_rec, k_rate, k_n = eng.tu_kernel_times()
    eng.kernel_timing(False)
    lw, lh = jobs['log2w'].astype(np.int64), jobs['log2h'].astype(np.int64)
    # SURVEY.md 8d: a separable transform costs w*h*(w_out + h_out) MACs (64-point sides keep 32 outputs); forward + inverse
    macs = float((2 * (1 << (lw + lh)) * (np.minimum(1 << lw, 32) + np.minimum(1 << lh, 32))).sum())
    # CPU port on a bounded sample of the same jobs (prediction from the oracle's RMD pass, then the TU chain)
    sel = np.linspace(0, len(jobs) - 1, 4000).astype(int)
    t0 = time.perf_counter()
    _, _, preds = O.rmd_batch(frame, frame, BITS, CTU, vis[sel], want_pred=True)
    for k, i in enumerate(sel):
        j = jobs[i]
        w, h = 1 << int(j['log2w']), 1 << int(j['log2h'])
        p = preds[k][int(src[i]['slot'])]
        r = (frame[int(j['y']):int(j['y']) + h, int(j['x']):int(j['x']) + w].astype(np.int32) - p).astype(np.int16)
        qp = 6 * int(j['qp_per']) + int(j['qp_rem'])
        co = O.fwd_transform(r, BITS, 0)
        lvl, _ = O.dep_quant(co, BITS, 0, 0, qp, float(j['lambda']), rates[0], 0)
        O.inv_transform(O.dep_dequant(lvl, BITS, qp), BITS, 0)
        O.residual_bits(lvl, 0, w <= 32 and h <= 32, w <= 32 and h <= 32, 1, states[0])
    cpu_s = time.perf_counter() - t0
    kern_ms = (k_tr + k_dq + k_rec + k_rate) / max(1, k_n)
    return {'workload': 'frame 0, the best rough-mode-decision candidate of every candidate CU (%d TUs, %d samples): prediction, residual, DCT-II, '
                        'dependent quantisation, inverse, reconstruction, SSE, residual bits; QP 32' % (len(jobs), n_samples),
            'tus_per_s_kernels': len(jobs) / (kern_ms * 1e-3) if kern_ms else None,
            'tus_per_s_e2e': len(jobs) / wall,
            'kernel_ms': {'predict_transform': k_tr / max(1, k_n), 'dep_quant': k_dq / max(1, k_n), 'reconstruct': k_rec / max(1, k_n), 'residual_bits': k_rate / max(1, k_n),
                          'note': 'events around the launches of vvcb_tu_eval_pred: prediction + transform pass, first-position + sort + dependent quantisation, reconstruction pass'},
            'e2e_ms': wall * 1e3, 'h2d_bytes': int(vis.nbytes + src.nbytes + jobs.nbytes), 'd2h_bytes': int(out['results'].nbytes),
            'transform_gmacs_per_s': macs / (((k_tr + k_rec) / max(1, k_n)) * 1e-3) / 1e9 if k_n else None,
            'transform_int_alu_frac': (macs / (((k_tr + k_rec) / max(1, k_n)) * 1e-3) / 1e9) / int_peak[0] if k_n and int_peak[0] else None,
            'nonzero_tu_fraction': float((out['results']['abs_sum_level'] > 0).mean()),
            'mean_residual_bits': float(out['results']['frac_bits'].mean() / 32768.0),
            'cpu_baseline': {'value': len(sel) / cpu_s, 'unit': 'TU/s', 'cores': 1, 'kind': 'port',
                             'sample': 'oracle: all predictions of the visit (its RMD pass) + transform + dependent quantisation + inverse + residual bits on %d of the jobs, %.1f s' % (len(sel), cpu_s)}}


def cpu_baseline_port(base, frame):
    """The oracle (plain-C port of the same sweep) on one host core, on the visits of the first two CTUs."""
    from oracle import oracle_py as O
    sel = base[base['y'] < 256]                          # the first two CTU rows of the frame: 30 CTUs
    t0 = time.perf_counter()
    O.rmd_batch(frame, frame, BITS, CTU, sel)
    dt = time.perf_counter() - t0
    return {'value': 30.0 / dt, 'unit': 'CTU/s', 'cores': 1, 'kind': 'port',
            'sample': 'oracle/vvc_oracle.c, same exhaustive sweep, the %d visits of the first two CTU rows (30 CTUs) of frame 0, %.1f s' % (len(sel), dt)}


def write_crop(d, frames, k):
    """Input of walker k: a 128x128 10-bit crop (1 CTU) of the synthetic frames with flat chroma -- the same crops the reference arm encodes."""
    crops = [(cx, cy) for cy in range(0, H - CTU + 1, CTU) for cx in range(0, W - CTU + 1, CTU)]
    cx, cy = crops[(7 * k) % len(crops)]
    os.makedirs(d, exist_ok=True)
    y = frames[k % NFRAMES][cy:cy + CTU, cx:cx + CTU].astype('<u2')
    c = np.full((CTU // 2, CTU // 2), 512, '<u2')
    open(os.path.join(d, 'in.yuv'), 'wb').write(y.tobytes() + c.tobytes() + c.tobytes())
    open(os.path.join(d, 'Time_python.dat'), 'w').close()


def encoder_cmd(enc, cfg, qp, out):
    # VVCB_BENCH_ENCODER_ARGS: extra reference-encoder options for side experiments (both arms get them), e.g. "--ALF=0"
    return [enc, '-c', cfg, '-i', 'in.yuv', '-wdt', str(CTU), '-hgt', str(CTU), '-q', str(qp), '-f', '1', '-fr', '30', '-b', out,
            '--InputBitDepth=10', '--InternalBitDepth=10', '--OutputBitDepth=10'] + os.environ.get('VVCB_BENCH_ENCODER_ARGS', '').split()


def bitexact_leg(frames, device):
    """The bit-exact use of the engine, measured like for like (SURVEY.md 7.2 option A): N walker processes -- the UNMODIFIED reference
    encoder with its luma intra cost evaluation served by the engine (oracle/_ref/EncoderAppServe), one 128x128 10-bit CTU crop each,
    QP cycling 22/27/32/37 -- share ONE engine context through the broker (vvc_intra_b200/vvcb_broker); next to it the plain reference
    encoder on the same crops and the same host cores.  Every served bitstream must equal the plain one byte for byte."""
    ref = os.path.join(ROOT, 'oracle/_ref')
    plain, served, cfg = (os.path.join(ref, f) for f in ('EncoderApp', 'EncoderAppServe', 'encoder_intra.cfg'))
    broker = os.environ.get('VVCB_BENCH_BROKER') or os.path.join(ROOT, 'vvc_intra_b200/vvcb_broker')     # override: development against the CPU stand-in
    if not all(os.path.exists(p) for p in (plain, served, cfg, broker)):
        return {'unavailable': 'oracle/_ref/EncoderAppServe or vvc_intra_b200/vvcb_broker was not built (run __graft_entry__.build() in the container that has /root/reference)'}
    cores = max(1, min(os.cpu_count() or 1, 64))
    # walkers per host core and broker worker threads: the setting that measured best (profiles/r2_bitexact_scaling.json) -- the walkers'
    # own CPU time bounds the leg from 256 walkers on 16 cores on, and two workers keep the batches large (about 30 CUs each)
    over = max(1, int(os.environ.get('VVCB_BENCH_OVERSUBSCRIBE', '16')))
    workers = max(1, int(os.environ.get('VVCB_BENCH_WORKERS', '2')))
    n = min(cores * over, 512)                       # bounded: a 6 MB broker slot and one encoder process per walker
    # the plain encoder runs on a bounded share of the same crops (its rate does not depend on how many there are); those are the
    # bitstreams the served ones are compared with
    n_plain = min(n, cores * max(1, int(os.environ.get('VVCB_BENCH_PLAIN_ROUNDS', '2'))))
    tmp = tempfile.mkdtemp(prefix='vvcbit_')
    env = dict(os.environ)
    env.pop('VVCB_BROKER', None)
    qps = [QPS[k % len(QPS)] for k in range(n)]
    for k in range(n):
        write_crop(os.path.join(tmp, 'w%d' % k), frames, k)
    # plain reference: `cores` processes at a time
    t0 = time.perf_counter()
    for base in range(0, n_plain, cores):
        procs = [subprocess.Popen(encoder_cmd(plain, cfg, qps[k], 'plain.bin'), cwd=os.path.join(tmp, 'w%d' % k), env=env, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
                 for k in range(base, min(n_plain, base + cores))]
        if any(p.wait() for p in procs):
            raise SystemExit('bench: the plain reference encoder failed')
    plain_s = time.perf_counter() - t0
    # served: all walkers at once behind one broker (they sleep while the engine works, so more walkers than cores keep the cores busy)
    path = os.path.join(tmp, 'broker.shm')
    server = subprocess.Popen([broker, path, '--device', str(device), '--bit-depth', '10', '--clients', str(n), '--frame', '%dx%d' % (CTU, CTU), '--workers', str(workers)], env=env,
                              stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
    try:
        for _ in range(1200):
            if os.path.exists(path) or server.poll() is not None:
                break
            time.sleep(0.05)
        if server.poll() is not None:
            raise SystemExit('bench: the broker did not start: ' + server.stderr.read()[-500:])
        t0 = time.perf_counter()
        procs = [subprocess.Popen(encoder_cmd(served, cfg, qps[k], 'served.bin'), cwd=os.path.join(tmp, 'w%d' % k),
                                  env=dict(env, VVCB_BROKER=path, VVCB_SHIM_REPORT=os.path.join(tmp, 'w%d' % k, 'report.json')), stdout=subprocess.DEVNULL, stderr=subprocess.PIPE, text=True)
                 for k in range(n)]
        for p in procs:
            _, err = p.communicate()
            if p.returncode:
                raise SystemExit('bench: a served encoder failed: ' + err[-500:])
        served_s = time.perf_counter() - t0
        stats = json.loads(subprocess.check_output([broker, path, '--stats'], env=env))
    finally:
        subprocess.run([broker, path, '--stop'], env=env)
        try:
            server.wait(timeout=60)
        except subprocess.TimeoutExpired:
            server.kill()
    same = sum(open(os.path.join(tmp, 'w%d' % k, 'plain.bin'), 'rb').read() == open(os.path.join(tmp, 'w%d' % k, 'served.bin'), 'rb').read() for k in range(n_plain))
    if same != n_plain:
        raise SystemExit('bench: %d of %d served bitstreams differ from the plain reference encoder\'s' % (n_plain - same, n_plain))
    reps = [json.load(open(os.path.join(tmp, 'w%d' % k, 'report.json'))) for k in range(n)]
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)
    tot = lambda key: sum(r[key] for r in reps)
    return {'workload': '%d walkers = %d host cores x %d: 128x128 10-bit CTU crops of the synthetic 1080p frames, QP cycling 32/27/37/22, shipped cfg (all tools on); '
                        'full encode of the CTU (split search + full RD + chroma), luma whole-CU cost evaluation served by the engine through one broker context' % (n, cores, over),
            'ctus_per_s': n / served_s, 'plain_reference_ctus_per_s': n_plain / plain_s, 'ratio': (n / served_s) / (n_plain / plain_s), 'cores': cores, 'walkers': n, 'broker_workers': workers,
            'bitstreams_identical': same, 'bitstreams_compared': n_plain, 'seconds': {'served': served_s, 'plain': plain_s},
            'engine_busy_frac': stats['busy_ns'] / stats['wall_ns'] / workers if stats['wall_ns'] else None,
            'broker': {k: stats[k] for k in ('cycles', 'requests', 'visits', 'tu_jobs', 'max_batch', 'kernel_launches')},
            # host wall time of the workers inside vvcb_cu_eval per batch, microseconds: pack + launch the rough mode decision, wait for its
            # lists, expand the templates, launch the TU stage, wait for it, hand the outputs back; then the device spans of the two stages
            'batch_phase_us': [round(x / 1e3 / max(1, stats['cycles']), 1) for x in stats.get('phase_ns', [])],
            'mean_round_trips_merged_per_batch': stats['requests'] / max(1, stats['cycles']),
            'walker_wait_for_engine_s_mean': tot('engine_wait_s') / n,
            'served_calls': {k: tot(k) for k in ('visits', 'predictions_skipped', 'distortions_served', 'tu_quantised', 'tu_sse', 'tu_residual_bits', 'jobs_prefetched', 'demand_round_trips')},
            'note': 'like for like: same crops, same cores, same encoder binary objects; ISP sub-partitions, chroma and the split walk itself still run the reference code on the host '
                    '(about 60 % of its CPU time), which bounds the ratio (Amdahl); engine_busy_frac = share of wall time a broker worker thread spends inside engine calls (mean over the workers)'}


def run_reference(args, rank, world):
    if rank != 0:
        return
    enc = os.path.join(ROOT, 'oracle/_ref/EncoderApp')
    cfg = os.path.join(ROOT, 'oracle/_ref/encoder_intra.cfg')
    if not (os.path.exists(enc) and os.path.exists(cfg)):
        emit({'impl': 'reference', 'unavailable': 'oracle/_ref/EncoderApp was not built (run __graft_entry__.build() in the container that has /root/reference)'})
        return
    cores = max(1, min(os.cpu_count() or 1, 64))
    frames = [synth_luma(f) for f in range(NFRAMES)]
    tmp = tempfile.mkdtemp(prefix='vvcref_')
    crops = [(cx, cy) for cy in range(0, H - CTU + 1, CTU) for cx in range(0, W - CTU + 1, CTU)]

    def one_step(s):
        f, qp = s % NFRAMES, QPS[s % len(QPS)]
        procs = []
        for k in range(cores):
            cx, cy = crops[(s * cores + k) % len(crops)]
            d = os.path.join(tmp, 's%d_%d' % (s, k))
            os.makedirs(d, exist_ok=True)
            y = frames[f][cy:cy + CTU, cx:cx + CTU].astype('<u2')
            c = np.full((CTU // 2, CTU // 2), 512, '<u2')
            open(os.path.join(d, 'in.yuv'), 'wb').write(y.tobytes() + c.tobytes() + c.tobytes())
            open(os.path.join(d, 'Time_python.dat'), 'w').close()
            procs.append(subprocess.Popen([enc, '-c', cfg, '-i', 'in.yuv', '-wdt', str(CTU), '-hgt', str(CTU), '-q', str(qp), '-f', '1',
                                           '-fr', '30', '-b', 'out.bin', '--InputBitDepth=10', '--InternalBitDepth=10',
                                           '--OutputBitDepth=10'], cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL))
        rcs = [p.wait() for p in procs]
        if any(rcs):
            raise RuntimeError('reference encoder failed: %r' % rcs)

    for s in range(min(args.warmup, 1)):
        one_step(s)
    t0 = time.perf_counter()
    for s in range(args.steps):
        one_step(args.warmup + s)
    dt = time.perf_counter() - t0
    value = args.steps * cores / dt
    # BASELINE.json's second metric, like for like: the rough-mode-decision evaluations (one prediction + SAD + SATD each) the plain encoder
    # makes per CTU, counted by the pass-through twin (oracle/_ref/EncoderAppServe with VVCB_SHIM_OFF=1: every call runs the reference's own
    # code, the link-time wrappers only count) on one crop per QP, outside the timed region
    evals_per_ctu = None
    twin = os.path.join(ROOT, 'oracle/_ref/EncoderAppServe')
    if os.path.exists(twin):
        procs = []
        for k, qp in enumerate(QPS):
            d = os.path.join(tmp, 'count%d' % k)
            write_crop(d, frames, k)
            procs.append((d, subprocess.Popen(encoder_cmd(twin, cfg, qp, 'out.bin'), cwd=d, env=dict(os.environ, VVCB_SHIM_OFF='1', VVCB_SHIM_REPORT=os.path.join(d, 'report.json')),
                                              stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)))
        counts = []
        for d, pr in procs:
            if pr.wait() == 0 and os.path.exists(os.path.join(d, 'report.json')):
                counts.append(json.load(open(os.path.join(d, 'report.json')))['reference_satd_evals'])
        if counts:
            evals_per_ctu = sum(counts) / len(counts)
    sample = ('unmodified reference encoder (VTM 6.1 fork, encoder_intra.cfg, all tools on, AVX2 dispatch), one process per 128x128 '
              '10-bit crop (1 CTU) of the same synthetic frames, %d processes at a time, QP cycling 32/27/37/22; '
              'full encode of the CTU (split search + full RD), not only the RMD sweep' % cores)
    emit({
        'impl': 'reference',
        'metric': 'all-intra 1080p10 CTUs/sec (exhaustive RMD sweep: intra pred + SAD/SATD + mode cost + candidate lists)',
        'value': value, 'unit': 'CTU/s', 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt / args.steps * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'int16 samples / int32 arithmetic / f64 costs', 'data': 'synthetic',
        'config': {'workload': 'configs[1]: all-intra 1920x1080 10-bit synthetic YUV, 8 frames, QP 22/27/32/37 (bounded sample: %d CTU crops per step)' % cores},
        'cpu_baseline': {'value': value, 'unit': 'CTU/s', 'cores': cores, 'kind': 'reference', 'sample': sample},
        'e2e': {'value': value, 'unit': 'CTU/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'satd_evals_per_s': value * evals_per_ctu if evals_per_ctu else None,
        'satd_evals_per_ctu': evals_per_ctu,
        'satd_evals_note': 'rough-mode-decision evaluations (prediction + SAD + SATD of one mode of one CU) the plain encoder makes per CTU, counted on one crop per QP by the '
                           'pass-through twin; the b200 arm evaluates every slot of every candidate CU (satd_evals_per_step), the reference only the ones its pruned walk reaches',
    })
    import shutil
    shutil.rmtree(tmp, ignore_errors=True)


_JSON_OUT = None


def emit(obj):
    """The one JSON line of the contract, on the process's original stdout."""
    _JSON_OUT.write(json.dumps(obj) + '\n')
    _JSON_OUT.flush()


def main():
    global _JSON_OUT
    # stdout carries exactly one JSON line: libraries that chat on fd 1 (NCCL prints its version there) are sent to stderr
    _JSON_OUT = os.fdopen(os.dup(1), 'w')
    sys.stdout.flush()
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-tu-stage', action='store_true')
    ap.add_argument('--no-strong', action='store_true', help='skip the configs[2] strong-scaling leg (64 x 2160p frames sharded over the ranks)')
    ap.add_argument('--no-bitexact', action='store_true', help='skip the brokered bit-exact encode leg (walker processes + plain reference on the host cores)')
    ap.add_argument('--resident-only', action='store_true', help='profiling aid: only the HBM-resident timed loop (no e2e / TU / CPU legs); not a bench line')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the result records of the last timed step (a fixed sample of %d visits) as DIR/<field>.npy' % DUMP_VISITS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs applies to the b200 arm')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local_rank))
    run_b200(args, rank, world, local_rank, dist)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
