"""ctypes mirror of the C ABI in include/vvc_intra_b200.h (one method per entry point, same names, same
argument meaning, errors raised as EngineError with the library's message -- the reference throws
Exception, CL/TypeDef.h:1322).  No compute happens in Python and nothing here falls back to a CPU."""
import ctypes as C
import os

import numpy as np

NUM_SLOTS, MAX_LIST = 112, 16
SLOT_MRL1, SLOT_MRL3, SLOT_MIP = 67, 72, 77
SAT_NONE = 0xFFFFFFFF
VISIT_NO_MRL, VISIT_NO_MIP = 1, 2

# struct vvcb_rmd_visit / vvcb_rmd_result (include/vvc_intra_b200.h)
VISIT_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('log2w', 'u1'), ('log2h', 'u1'), ('avail_al', 'u1'),
                        ('n_above', 'u1'), ('n_above_right', 'u1'), ('n_left', 'u1'), ('n_below_left', 'u1'),
                        ('flags', 'u1'), ('mpm', 'u1', 6), ('num_mpm_cand', 'u1'), ('pad', 'u1', 3),
                        ('rates', '<u4', 11), ('sqrt_lambda', '<f8')], align=True)
MODE_DTYPE = np.dtype([('mip', 'u1'), ('mrl', 'u1'), ('mode', 'u1'), ('pad', 'u1')])


MAX_HAD_LIST = 8
RESULT_DTYPE = np.dtype([('n_rd', '<i4'), ('n_had', '<i4'), ('n_final', '<i4'), ('pad', '<i4'),
                         ('rd_mode', MODE_DTYPE, MAX_LIST), ('rd_cost', '<f8', MAX_LIST),
                         ('had_mode', MODE_DTYPE, MAX_HAD_LIST), ('had_cost', '<f8', MAX_HAD_LIST),
                         ('final_mode', MODE_DTYPE, MAX_LIST)], align=True)
DETAIL_DTYPE = np.dtype([('sad', '<u4', NUM_SLOTS), ('satd', '<u4', NUM_SLOTS), ('n_reg', '<i4'), ('n_reg_had', '<i4'),
                         ('reg_mode', MODE_DTYPE, MAX_LIST), ('reg_cost', '<f8', MAX_LIST),
                         ('reg_had_mode', MODE_DTYPE, MAX_HAD_LIST), ('reg_had_cost', '<f8', MAX_HAD_LIST)], align=True)
assert VISIT_DTYPE.itemsize == 80 and RESULT_DTYPE.itemsize == 368 and DETAIL_DTYPE.itemsize == 1192, \
    (VISIT_DTYPE.itemsize, RESULT_DTYPE.itemsize, DETAIL_DTYPE.itemsize)


OPT_DEP_QUANT = 1
TU_QUANT, TU_DEPQUANT, TU_RDOQ_TS, TU_TS_ALLOWED, TU_MTS_ALLOWED, TU_RATE = 1, 2, 4, 8, 16, 32
BIN_MODEL_DTYPE = np.dtype([('state', '<u2', 2), ('rate', 'u1'), ('pad', 'u1')])
CTX_STATES_DTYPE = np.dtype([('mts_idx', BIN_MODEL_DTYPE, 11), ('sig_sbb', BIN_MODEL_DTYPE, 2), ('sig', BIN_MODEL_DTYPE, (3, 12)), ('par', BIN_MODEL_DTYPE, 21),
                             ('gt1', BIN_MODEL_DTYPE, 21), ('gt2', BIN_MODEL_DTYPE, 21), ('last_x', BIN_MODEL_DTYPE, 20), ('last_y', BIN_MODEL_DTYPE, 20),
                             ('ts_sig_sbb', BIN_MODEL_DTYPE, 3), ('ts_sig', BIN_MODEL_DTYPE, 3), ('ts_par', BIN_MODEL_DTYPE, 1), ('ts_gtx', BIN_MODEL_DTYPE, 5),
                             ('ts_lrg1', BIN_MODEL_DTYPE, 4), ('ts_sign', BIN_MODEL_DTYPE, 6)])
TU_JOB_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('log2w', 'u1'), ('log2h', 'u1'), ('mts_idx', 'u1'), ('flags', 'u1'),
                         ('qp_per', '<i2'), ('qp_rem', '<i2'), ('offset', '<u4'), ('rate_idx', '<u2'), ('lfnst_idx', 'u1'), ('intra_mode', 'u1'),
                         ('cbf_delta_bits', '<i4'), ('lambda', '<f8')], align=True)
TU_RESULT_DTYPE = np.dtype([('abs_sum_coeff', '<i4'), ('abs_sum_level', '<i4'), ('sse', '<u8'), ('frac_bits', '<u8')], align=True)
TU_SRC_DTYPE = np.dtype([('visit', '<u4'), ('slot', 'u1'), ('pad', 'u1', 3)])
DQ_RATES_DTYPE = np.dtype([('sig_sbb', '<u4', (2, 2)), ('sig', '<u4', (3, 12, 2)), ('par', '<u4', (21, 2)), ('gt1', '<u4', (21, 2)),
                           ('gt2', '<u4', (21, 2)), ('last_x', '<u4', (20, 2)), ('last_y', '<u4', (20, 2)),
                           ('ts_sig_sbb', '<u4', (3, 2)), ('ts_sig', '<u4', (3, 2)), ('ts_par', '<u4', (1, 2)), ('ts_gtx', '<u4', (5, 2)),
                           ('ts_lrg1', '<u4', (4, 2)), ('ts_sign', '<u4', (6, 2))])
assert TU_SRC_DTYPE.itemsize == 8 and TU_JOB_DTYPE.itemsize == 32 and TU_RESULT_DTYPE.itemsize == 24 and CTX_STATES_DTYPE.itemsize == 1044 and DQ_RATES_DTYPE.itemsize == 1304


FEAT_CU_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('w', 'u1'), ('h', 'u1'), ('qt_depth', 'u1'), ('mt_depth', 'u1')])
FEAT_JOB_DTYPE = np.dtype([('cu', FEAT_CU_DTYPE), ('n_neighbours', 'u1'), ('pad', 'u1', 7), ('nb', FEAT_CU_DTYPE, 5)])
FEAT_RESULT_DTYPE = np.dtype([('f', '<i4', 27), ('valid', '<i4')])
assert FEAT_JOB_DTYPE.itemsize == 56 and FEAT_RESULT_DTYPE.itemsize == 112


BRIEF_DTYPE = np.dtype([('n_rd', 'u1'), ('n_had', 'u1'), ('n_final', 'u1'), ('pad', 'u1'), ('final_mode', '<u2', MAX_LIST), ('had_mode', '<u2', MAX_HAD_LIST), ('reserved', 'u1', 12)])
assert BRIEF_DTYPE.itemsize == 64
OPT_YIELD_SYNC, OPT_TRUSTED_VISITS = 2, 3
RECT_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('w', '<i2'), ('h', '<i2'), ('offset', '<u4')])
assert RECT_DTYPE.itemsize == 12


class CuRequest(C.Structure):
    """struct vvcb_cu_request: one CU of a host walk (rectangles to push, the visit, TU candidates, output pointers)."""
    _fields_ = [('rects', C.c_void_p), ('n_rects', C.c_int), ('rect_samples', C.c_void_p), ('n_rect_samples', C.c_size_t),
                ('visit', C.c_void_p), ('want_rmd', C.c_int), ('jobs', C.c_void_p), ('slots', C.c_void_p), ('n_jobs', C.c_int),
                ('rates', C.c_void_p), ('states', C.c_void_p), ('result', C.c_void_p), ('detail', C.c_void_p),
                ('level', C.c_void_p), ('reco', C.c_void_p), ('pred', C.c_void_p), ('tu_results', C.c_void_p),
                ('autos', C.c_void_p), ('n_autos', C.c_int), ('max_auto', C.c_int), ('n_auto', C.c_void_p), ('auto_slot', C.c_void_p), ('auto_tmpl', C.c_void_p),
                ('auto_level', C.c_void_p), ('auto_reco', C.c_void_p), ('auto_pred', C.c_void_p), ('auto_results', C.c_void_p)]


CU_AUTO_DTYPE = np.dtype([('job', TU_JOB_DTYPE), ('modes', 'u1'), ('skip_mip', 'u1'), ('pad', 'u1', 6)])
# vvcb_isp_part (include/vvc_intra_b200.h): one transform block of an intra sub-partition CU
ISP_PART_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('w', '<i2'), ('h', '<i2'), ('pred_x', '<i2'), ('pred_y', '<i2'), ('pred_w', '<i2'), ('pred_h', '<i2'),
                           ('top_ref_len', '<i2'), ('left_ref_len', '<i2'), ('fetch_top_len', '<i2'), ('fetch_left_len', '<i2'),
                           ('predicts', 'u1'), ('tr_hor', 'u1'), ('tr_ver', 'u1'), ('last', 'u1')])
ISP_MODE_DTYPE = np.dtype([('angle', '<i2'), ('inv_angle', '<u2'), ('is_ver', 'u1'), ('pdpc', 'u1'), ('ang_scale', 'i1'), ('pad', 'u1')])
ISP_HOR, ISP_VER, TR_DCT2, TR_DCT8, TR_DST7 = 1, 2, 0, 1, 2
assert CU_AUTO_DTYPE.itemsize == 40
# vvcb_isp_job / vvcb_isp_result (include/vvc_intra_b200.h): one ISP candidate and its per-block results
ISP_JOB_DTYPE = np.dtype([('visit', '<u4'), ('isp_mode', 'u1'), ('mode', 'u1'), ('flags', 'u1'), ('use_mts', 'u1'), ('max_tb_size', 'u1'),
                          ('lfnst_idx', 'u1'), ('qp_per', '<i2'), ('qp_rem', '<i2'), ('rate_idx', '<u2'), ('offset', '<u4'),
                          ('cbf', BIN_MODEL_DTYPE, 2), ('lambda', '<f8')], align=True)
ISP_MAX_PARTS = 4
ISP_RESULT_DTYPE = np.dtype([('part', TU_RESULT_DTYPE, ISP_MAX_PARTS), ('cbf_bits', '<u4', ISP_MAX_PARTS), ('cbf', 'u1', ISP_MAX_PARTS),
                             ('n_parts', 'u1'), ('discarded', 'u1'), ('pad', 'u1', 2)], align=True)
assert ISP_JOB_DTYPE.itemsize == 40 and ISP_RESULT_DTYPE.itemsize == 120
AUTO_FINAL, AUTO_REGULAR = 1, 2
# vvcb_chroma_visit / vvcb_chroma_result (include/vvc_intra_b200.h): one chroma CU of the separate tree, its 8 candidates' distortions
CHROMA_CANDS, LM_CHROMA, MDLM_L, MDLM_T, DM_CHROMA = 8, 67, 68, 69, 70
CHROMA_VISIT_DTYPE = np.dtype([('x', '<i2'), ('y', '<i2'), ('log2w', 'u1'), ('log2h', 'u1'), ('avail_al', 'u1'), ('n_above', 'u1'),
                               ('n_above_right', 'u1'), ('n_left', 'u1'), ('n_below_left', 'u1'), ('dm_mode', 'u1'), ('cclm', 'u1'), ('pad', 'u1', 3)])
CHROMA_RESULT_DTYPE = np.dtype([('mode', 'u1', CHROMA_CANDS), ('sad', '<u4', (CHROMA_CANDS, 2)), ('satd', '<u4', (CHROMA_CANDS, 2))], align=True)
assert CHROMA_VISIT_DTYPE.itemsize == 16 and CHROMA_RESULT_DTYPE.itemsize == 136
# vvcb_chroma_ctx_states / vvcb_chroma_tu_job / vvcb_chroma_tu_result (include/vvc_intra_b200.h): chroma TU coding of the candidates
CHROMA_CTX_STATES_DTYPE = np.dtype([('cbf_cb', BIN_MODEL_DTYPE, 2), ('cbf_cr', BIN_MODEL_DTYPE, 3), ('sig_sbb', BIN_MODEL_DTYPE, 2),
                                    ('sig', BIN_MODEL_DTYPE, (3, 8)), ('par', BIN_MODEL_DTYPE, 11), ('gt1', BIN_MODEL_DTYPE, 11),
                                    ('gt2', BIN_MODEL_DTYPE, 11), ('last_x', BIN_MODEL_DTYPE, 3), ('last_y', BIN_MODEL_DTYPE, 3)])
CHROMA_TU_JOB_DTYPE = np.dtype([('visit', '<u4'), ('cand', 'u1'), ('flags', 'u1'), ('rate_idx', '<u2'), ('qp_per', '<i2', 2), ('qp_rem', '<i2', 2),
                                ('offset', '<u4'), ('pad', '<u4'), ('lambda', '<f8', 2)], align=True)
CHROMA_TU_RESULT_DTYPE = np.dtype([('comp', TU_RESULT_DTYPE, 2), ('cbf_bits', '<u4', 2), ('cbf', 'u1', 2), ('pad', 'u1', 6)], align=True)
assert CHROMA_CTX_STATES_DTYPE.itemsize == 420 and CHROMA_TU_JOB_DTYPE.itemsize == 40 and CHROMA_TU_RESULT_DTYPE.itemsize == 64
# vvcb_chroma_joint_ctx_states / vvcb_chroma_joint_tu_job / vvcb_chroma_joint_tu_result (include/vvc_intra_b200.h): joint Cb-Cr candidates
CHROMA_JOINT_CTX_STATES_DTYPE = np.dtype([('chroma', CHROMA_CTX_STATES_DTYPE), ('joint', BIN_MODEL_DTYPE, 3)])
CHROMA_JOINT_TU_JOB_DTYPE = np.dtype([('visit', '<u4'), ('cand', 'u1'), ('flags', 'u1'), ('rate_idx', '<u2'), ('mode', 'u1'), ('sign', 'i1'),
                                      ('qp_per', '<i2'), ('qp_rem', '<i2'), ('pad', '<u2'), ('offset', '<u4'), ('pad2', '<u4'), ('lambda', '<f8')],
                                     align=True)
CHROMA_JOINT_TU_RESULT_DTYPE = np.dtype([('res', TU_RESULT_DTYPE), ('sse', '<u8', 2), ('cbf_bits', '<u4', 2), ('joint_bits', '<u4'), ('cbf', 'u1'),
                                         ('pad', 'u1', 3)], align=True)
assert CHROMA_JOINT_CTX_STATES_DTYPE.itemsize == 438 and CHROMA_JOINT_TU_JOB_DTYPE.itemsize == 32 and CHROMA_JOINT_TU_RESULT_DTYPE.itemsize == 56


class EngineError(RuntimeError):
    pass


def library_path():
    # VVCB_LIBRARY_PATH: developer override used to A/B kernel build variants (tools/variants.sh)
    return os.environ.get('VVCB_LIBRARY_PATH') or os.path.join(os.path.dirname(os.path.abspath(__file__)), 'libvvc_intra_b200.so')


_lib = None


def load_library():
    """Loads libvvc_intra_b200.so; fails loudly when the CUDA extension has not been built."""
    global _lib
    if _lib is None:
        path = library_path()
        if not os.path.exists(path):
            raise EngineError('%s is missing: run `python -c "import __graft_entry__ as g; g.build()"` '
                              '(there is no CPU fallback)' % path)
        L = C.CDLL(path)
        L.vvcb_last_error.restype = C.c_char_p
        L.vvcb_last_error.argtypes = [C.c_void_p]
        L.vvcb_launch_count.restype = C.c_uint64
        L.vvcb_launch_count.argtypes = [C.c_void_p]
        L.vvcb_create.argtypes = [C.POINTER(C.c_void_p), C.c_int, C.c_int, C.c_int]
        L.vvcb_destroy.argtypes = [C.c_void_p]
        L.vvcb_destroy.restype = None
        L.vvcb_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.vvcb_frame_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.vvcb_reco_update.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.vvcb_rmd_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.vvcb_rmd_eval_brief.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.vvcb_rmd_eval_brief_resident.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.vvcb_rmd_eval_device.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.vvcb_rmd_pred.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.vvcb_rmd_pred_all.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_dev_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.vvcb_dev_free.argtypes = [C.c_void_p, C.c_void_p]
        L.vvcb_host_alloc.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(C.c_void_p)]
        L.vvcb_host_free.argtypes = [C.c_void_p, C.c_void_p]
        L.vvcb_dev_upload.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.vvcb_dev_download.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]
        L.vvcb_sync.argtypes = [C.c_void_p]
        L.vvcb_tu_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_tu_eval_pred.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_int,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_residual_bits.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p]
        L.vvcb_mts_preselect.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.vvcb_mts_preselect.restype = None
        L.vvcb_calc_rd_cost.argtypes = [C.c_double, C.c_uint64, C.c_uint64]
        L.vvcb_calc_rd_cost.restype = C.c_double
        L.vvcb_isp_plan.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.vvcb_isp_mode_param.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
        L.vvcb_isp_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t,
                                    C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_chroma_frame_begin.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.vvcb_chroma_reco_update.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.vvcb_chroma_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.vvcb_chroma_tu_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_chroma_joint_tu_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_size_t,
                                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        L.vvcb_ctu_hads_islice.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.vvcb_features_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
        L.vvcb_frame_bind_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]
        L.vvcb_kernel_timing.argtypes = [C.c_void_p, C.c_int]
        L.vvcb_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        L.vvcb_tu_kernel_times.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int)]
        L.vvcb_cu_eval_phases.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.vvcb_measure_int_peak.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
        L.vvcb_frame_alloc.argtypes = [C.c_void_p, C.c_int, C.c_int]
        L.vvcb_reco_from_orig.argtypes = [C.c_void_p]
        L.vvcb_orig_update.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.vvcb_reco_update_rects.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t]
        L.vvcb_cu_eval.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        L.vvcb_broker_serve.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        L.vvcb_frame_share.argtypes = [C.c_void_p, C.c_void_p]
        L.vvcb_broker_stop.argtypes = [C.c_char_p]
        L.vvcb_broker_read_stats.argtypes = [C.c_char_p, C.c_void_p]
        L.vvcb_timer_start.argtypes = [C.c_void_p]
        L.vvcb_timer_stop.argtypes = [C.c_void_p, C.POINTER(C.c_float)]
        _lib = L
    return _lib


def _ptr(a):
    return C.c_void_p(a.ctypes.data)


class IntraCostEngine:
    """One engine context (= one CUDA device + stream).  Mirrors vvcb_create .. vvcb_destroy."""

    def __init__(self, device=0, bit_depth=10, ctu_size=128):
        self._lib = load_library()
        self._ctx = C.c_void_p()
        rc = self._lib.vvcb_create(C.byref(self._ctx), device, bit_depth, ctu_size)
        if rc != 0:
            raise EngineError(self._lib.vvcb_last_error(None).decode())
        self.bit_depth, self.ctu_size, self.device = bit_depth, ctu_size, device

    def close(self):
        if getattr(self, '_ctx', None):
            for p in getattr(self, '_pinned', []):
                self._lib.vvcb_host_free(self._ctx, p)
            self._pinned = []
            self._lib.vvcb_destroy(self._ctx)
            self._ctx = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def _ck(self, rc):
        if rc != 0:
            raise EngineError('%s (status %d)' % (self._lib.vvcb_last_error(self._ctx).decode(), rc))

    def cu_eval_phases(self):
        """vvcb_cu_eval_phases: (ns[8], calls) -- cumulative host nanoseconds of the six phases of vvcb_cu_eval and the device spans of its two stages."""
        ns, calls = (C.c_uint64 * 8)(), C.c_uint64(0)
        self._ck(self._lib.vvcb_cu_eval_phases(self._ctx, ns, C.byref(calls)))
        return [int(x) for x in ns], int(calls.value)

    def set_option(self, option, value):
        self._ck(self._lib.vvcb_set_option(self._ctx, option, value))

    # ---- planes
    def frame_begin(self, orig):
        orig = np.ascontiguousarray(orig, np.int16)
        self._ck(self._lib.vvcb_frame_begin(self._ctx, _ptr(orig), orig.shape[1], orig.shape[1], orig.shape[0]))

    def reco_update(self, reco, x=0, y=0):
        reco = np.ascontiguousarray(reco, np.int16)
        self._ck(self._lib.vvcb_reco_update(self._ctx, _ptr(reco), reco.shape[1], x, y, reco.shape[1], reco.shape[0]))

    def reco_from_orig(self):
        """vvcb_reco_from_orig: reconstruction := original on the device (the exhaustive sweep's neighbours)."""
        self._ck(self._lib.vvcb_reco_from_orig(self._ctx))

    def frame_alloc(self, width, height):
        """vvcb_frame_alloc: cleared planes for several pictures side by side (what the broker keeps)."""
        self._ck(self._lib.vvcb_frame_alloc(self._ctx, width, height))

    def orig_update(self, orig, x=0, y=0):
        orig = np.ascontiguousarray(orig, np.int16)
        self._ck(self._lib.vvcb_orig_update(self._ctx, _ptr(orig), orig.shape[1], x, y, orig.shape[1], orig.shape[0]))

    def reco_update_rects(self, rects, samples):
        rects = np.ascontiguousarray(rects, RECT_DTYPE)
        samples = np.ascontiguousarray(samples, np.int16).ravel()
        self._ck(self._lib.vvcb_reco_update_rects(self._ctx, _ptr(rects), len(rects), _ptr(samples), samples.size))

    def cu_eval(self, requests):
        """vvcb_cu_eval.  requests: list of dicts with optional keys rects (RECT_DTYPE) + rect_samples, visit (VISIT_DTYPE, 1 entry),
        want_rmd, jobs (TU_JOB_DTYPE) + slots (uint8) [+ rates (DQ_RATES_DTYPE, 1), states (CTX_STATES_DTYPE, 1)], autos (CU_AUTO_DTYPE templates,
        with want_rmd) + max_auto.  Returns a list of dicts: result / detail (want_rmd), level / reco / pred / tu_results (jobs), n_auto / auto_slot /
        auto_tmpl / auto_level / auto_reco / auto_pred / auto_results (templates)."""
        arr = (CuRequest * len(requests))()
        keep, outs = [], []
        for r, q in zip(arr, requests):
            o = {}
            if q.get('rects') is not None and len(q['rects']):
                rc = np.ascontiguousarray(q['rects'], RECT_DTYPE)
                sm = np.ascontiguousarray(q['rect_samples'], np.int16).ravel()
                keep += [rc, sm]
                r.rects, r.n_rects, r.rect_samples, r.n_rect_samples = rc.ctypes.data, len(rc), sm.ctypes.data, sm.size
            if q.get('visit') is not None:
                v = np.ascontiguousarray(q['visit'], VISIT_DTYPE).reshape(1)
                keep.append(v)
                r.visit = v.ctypes.data
                bs = 1 << (int(v['log2w'][0]) + int(v['log2h'][0]))
            if q.get('want_rmd'):
                o['result'], o['detail'] = np.zeros(1, RESULT_DTYPE), np.zeros(1, DETAIL_DTYPE)
                r.want_rmd, r.result, r.detail = 1, o['result'].ctypes.data, o['detail'].ctypes.data
            if q.get('jobs') is not None and len(q['jobs']):
                jb = np.ascontiguousarray(q['jobs'], TU_JOB_DTYPE)
                sl = np.ascontiguousarray(q['slots'], np.uint8)
                keep += [jb, sl]
                r.jobs, r.slots, r.n_jobs = jb.ctypes.data, sl.ctypes.data, len(jb)
                for key, dt in (('rates', DQ_RATES_DTYPE), ('states', CTX_STATES_DTYPE)):
                    if q.get(key) is not None:
                        a = np.ascontiguousarray(q[key], dt).reshape(1)
                        keep.append(a)
                        setattr(r, key, a.ctypes.data)
                o['level'], o['reco'], o['pred'] = np.zeros(len(jb) * bs, np.int32), np.zeros(len(jb) * bs, np.int16), np.zeros(len(jb) * bs, np.int16)
                o['tu_results'] = np.zeros(len(jb), TU_RESULT_DTYPE)
                r.level, r.reco, r.pred, r.tu_results = o['level'].ctypes.data, o['reco'].ctypes.data, o['pred'].ctypes.data, o['tu_results'].ctypes.data
            if q.get('autos') is not None and len(q['autos']):
                au = np.ascontiguousarray(q['autos'], CU_AUTO_DTYPE)
                mx = int(q.get('max_auto', 96))
                keep.append(au)
                for key, dt in (('rates', DQ_RATES_DTYPE), ('states', CTX_STATES_DTYPE)):
                    if q.get(key) is not None and not getattr(r, key):
                        a = np.ascontiguousarray(q[key], dt).reshape(1)
                        keep.append(a)
                        setattr(r, key, a.ctypes.data)
                o['n_auto'], o['auto_slot'], o['auto_tmpl'] = np.zeros(1, np.int32), np.zeros(mx, np.uint8), np.zeros(mx, np.uint8)
                o['auto_level'], o['auto_reco'], o['auto_pred'] = np.zeros(mx * bs, np.int32), np.zeros(mx * bs, np.int16), np.zeros(mx * bs, np.int16)
                o['auto_results'] = np.zeros(mx, TU_RESULT_DTYPE)
                r.autos, r.n_autos, r.max_auto, r.n_auto = au.ctypes.data, len(au), mx, o['n_auto'].ctypes.data
                r.auto_slot, r.auto_tmpl, r.auto_level, r.auto_reco = o['auto_slot'].ctypes.data, o['auto_tmpl'].ctypes.data, o['auto_level'].ctypes.data, o['auto_reco'].ctypes.data
                r.auto_pred, r.auto_results = o['auto_pred'].ctypes.data, o['auto_results'].ctypes.data
            outs.append(o)
        self._ck(self._lib.vvcb_cu_eval(self._ctx, C.byref(arr), len(requests)))
        return outs

    def frame_bind_device(self, d_orig, d_reco, stride, width, height):
        self._ck(self._lib.vvcb_frame_bind_device(self._ctx, d_orig, d_reco, stride, width, height))

    def kernel_timing(self, on=True):
        self._ck(self._lib.vvcb_kernel_timing(self._ctx, int(on)))

    def kernel_times(self):
        """(ms_plan, ms_eval, ms_lists, timed launches) accumulated since the last call."""
        ms = (C.c_float * 3)()
        n = C.c_int()
        self._ck(self._lib.vvcb_kernel_times(self._ctx, ms, C.byref(n)))
        return ms[0], ms[1], ms[2], n.value

    def tu_kernel_times(self):
        """(ms prediction + transform pass, ms quantiser kernels, ms reconstruction pass, ms rate estimation, timed calls)."""
        ms = (C.c_float * 4)()
        n = C.c_int()
        self._ck(self._lib.vvcb_tu_kernel_times(self._ctx, ms, C.byref(n)))
        return ms[0], ms[1], ms[2], ms[3], n.value

    # ---- rough mode decision
    def rmd_eval(self, visits, out=None, detail=False, detail_out=None):
        """vvcb_rmd_eval.  Returns the result array, or (results, details) when detail is requested."""
        visits = np.ascontiguousarray(visits, VISIT_DTYPE)
        if out is None:
            out = np.empty(len(visits), RESULT_DTYPE)
        elif out.dtype != RESULT_DTYPE or len(out) < len(visits) or not out.flags['C_CONTIGUOUS']:
            raise ValueError('out must be a contiguous RESULT_DTYPE array of at least len(visits) records')
        if detail and detail_out is None:
            detail_out = np.empty(len(visits), DETAIL_DTYPE)
        if detail_out is not None and (detail_out.dtype != DETAIL_DTYPE or len(detail_out) < len(visits) or not detail_out.flags['C_CONTIGUOUS']):
            raise ValueError('detail_out must be a contiguous DETAIL_DTYPE array of at least len(visits) records')
        self._ck(self._lib.vvcb_rmd_eval(self._ctx, _ptr(visits), len(visits), _ptr(out),
                                         _ptr(detail_out) if detail_out is not None else None))
        return (out, detail_out) if detail_out is not None else out

    def rmd_eval_brief(self, visits, out=None):
        """vvcb_rmd_eval_brief: 64-byte records (mode codes of the final and Hadamard lists)."""
        visits = np.ascontiguousarray(visits, VISIT_DTYPE)
        if out is None:
            out = np.empty(len(visits), BRIEF_DTYPE)
        elif out.dtype != BRIEF_DTYPE or len(out) < len(visits) or not out.flags['C_CONTIGUOUS']:
            raise ValueError('out must be a contiguous BRIEF_DTYPE array of at least len(visits) records')
        self._ck(self._lib.vvcb_rmd_eval_brief(self._ctx, _ptr(visits), len(visits), _ptr(out)))
        return out

    def rmd_eval_brief_resident(self, d_visits, n, out):
        """vvcb_rmd_eval_brief_resident: visits resident on the device (dev_alloc + dev_upload), brief records to the host array `out`."""
        if out.dtype != BRIEF_DTYPE or len(out) < n or not out.flags['C_CONTIGUOUS']:
            raise ValueError('out must be a contiguous BRIEF_DTYPE array of at least n records')
        self._ck(self._lib.vvcb_rmd_eval_brief_resident(self._ctx, d_visits, n, _ptr(out)))
        return out

    def rmd_pred(self, visit, slot):
        visit = np.ascontiguousarray(visit, VISIT_DTYPE).reshape(1)
        w, h = 1 << int(visit[0]['log2w']), 1 << int(visit[0]['log2h'])
        pred = np.zeros((h, w), np.int16)
        self._ck(self._lib.vvcb_rmd_pred(self._ctx, _ptr(visit), slot, _ptr(pred)))
        return pred

    def rmd_pred_all(self, visit):
        """vvcb_rmd_pred_all: (NUM_SLOTS, h, w) prediction samples of one visit."""
        visit = np.ascontiguousarray(visit, VISIT_DTYPE).reshape(1)
        w, h = 1 << int(visit['log2w'][0]), 1 << int(visit['log2h'][0])
        pred = np.zeros((NUM_SLOTS, h, w), np.int16)
        self._ck(self._lib.vvcb_rmd_pred_all(self._ctx, _ptr(visit), _ptr(pred)))
        return pred

    # ---- TU coding
    @staticmethod
    def _snapshots(rates, states):
        """Context prices (DQ_RATES_DTYPE) and context states (CTX_STATES_DTYPE) are parallel arrays indexed by job['rate_idx']."""
        rates = None if rates is None else np.ascontiguousarray(rates, DQ_RATES_DTYPE)
        states = None if states is None else np.ascontiguousarray(states, CTX_STATES_DTYPE)
        if rates is not None and states is not None and len(rates) != len(states):
            raise ValueError('rates and states must have the same length')
        nr = len(rates) if rates is not None else (len(states) if states is not None else 0)
        return rates, states, nr

    def tu_eval(self, jobs, resi, pred=None, want_coeff=False, want_level=False, want_reco=False, rates=None, states=None):
        """vvcb_tu_eval.  resi / pred: flat int16 arrays indexed by job['offset']; rates: DQ_RATES_DTYPE array indexed by
        job['rate_idx'] (jobs flagged TU_DEPQUANT).  Returns dict of outputs."""
        jobs = np.ascontiguousarray(jobs, TU_JOB_DTYPE)
        resi = np.ascontiguousarray(resi, np.int16).ravel()
        pred = None if pred is None else np.ascontiguousarray(pred, np.int16).ravel()
        ns = resi.size
        out = dict(results=np.zeros(len(jobs), TU_RESULT_DTYPE))
        if want_coeff:
            out['coeff'] = np.zeros(ns, np.int32)
        if want_level:
            out['level'] = np.zeros(ns, np.int32)
        if want_reco:
            out['reco'] = np.zeros(ns, np.int16)
        rates, states, nr = self._snapshots(rates, states)
        self._ck(self._lib.vvcb_tu_eval(self._ctx, _ptr(jobs), len(jobs), _ptr(resi), _ptr(pred) if pred is not None else None, ns,
                                        _ptr(rates) if rates is not None else None, _ptr(states) if states is not None else None, nr,
                                        _ptr(out['coeff']) if want_coeff else None, _ptr(out['level']) if want_level else None,
                                        _ptr(out['reco']) if want_reco else None, _ptr(out['results'])))
        return out

    def tu_eval_pred(self, visits, src, jobs, n_samples, want_coeff=False, want_level=False, want_reco=False, want_pred=False, rates=None, states=None):
        """vvcb_tu_eval_pred: prediction and residual are formed on the device from the frame planes (src: TU_SRC_DTYPE)."""
        visits = np.ascontiguousarray(visits, VISIT_DTYPE)
        src = np.ascontiguousarray(src, TU_SRC_DTYPE)
        jobs = np.ascontiguousarray(jobs, TU_JOB_DTYPE)
        out = dict(results=np.zeros(len(jobs), TU_RESULT_DTYPE))
        for key, want, dt in (('coeff', want_coeff, np.int32), ('level', want_level, np.int32), ('reco', want_reco, np.int16), ('pred', want_pred, np.int16)):
            if want:
                out[key] = np.zeros(n_samples, dt)
        rates, states, nr = self._snapshots(rates, states)
        p = lambda k: _ptr(out[k]) if k in out else None
        self._ck(self._lib.vvcb_tu_eval_pred(self._ctx, _ptr(visits), len(visits), _ptr(src), _ptr(jobs), len(jobs), n_samples,
                                             _ptr(rates) if rates is not None else None, _ptr(states) if states is not None else None, nr,
                                             p('coeff'), p('level'), p('reco'), p('pred'), _ptr(out['results'])))
        return out

    def isp_eval(self, visits, jobs, n_samples, states=None, want_level=False, want_reco=False, want_pred=False):
        """vvcb_isp_eval: ISP candidates (ISP_JOB_DTYPE) of the CUs in visits, blocks of at least 4x4.  states: CTX_STATES_DTYPE
        array indexed by job['rate_idx'].  Returns dict with 'results' (ISP_RESULT_DTYPE) and the wanted flat outputs of n_samples,
        each candidate's blocks in coding order at job['offset']."""
        visits = np.ascontiguousarray(visits, VISIT_DTYPE)
        jobs = np.ascontiguousarray(jobs, ISP_JOB_DTYPE)
        states = None if states is None else np.ascontiguousarray(states, CTX_STATES_DTYPE)
        out = dict(results=np.zeros(len(jobs), ISP_RESULT_DTYPE))
        for key, want, dt in (('level', want_level, np.int32), ('reco', want_reco, np.int16), ('pred', want_pred, np.int16)):
            if want:
                out[key] = np.zeros(n_samples, dt)
        p = lambda k: _ptr(out[k]) if k in out else None
        self._ck(self._lib.vvcb_isp_eval(self._ctx, _ptr(visits), len(visits), _ptr(jobs), len(jobs),
                                         _ptr(states) if states is not None else None, 0 if states is None else len(states), n_samples,
                                         p('level'), p('reco'), p('pred'), _ptr(out['results'])))
        return out

    # ---- chroma intra candidates (4:2:0)
    def chroma_frame_begin(self, cb, cr):
        """vvcb_chroma_frame_begin: Cb / Cr originals of the picture given to frame_begin (half its width and height); reconstructions cleared."""
        cb, cr = np.ascontiguousarray(cb, np.int16), np.ascontiguousarray(cr, np.int16)
        if cb.shape != cr.shape:
            raise ValueError('cb and cr must have the same shape')
        self._ck(self._lib.vvcb_chroma_frame_begin(self._ctx, _ptr(cb), _ptr(cr), cb.shape[1], cb.shape[1], cb.shape[0]))

    def chroma_reco_update(self, cb, cr, x=0, y=0):
        """vvcb_chroma_reco_update: the rectangle of both chroma reconstructions at (x, y), chroma samples."""
        cb, cr = np.ascontiguousarray(cb, np.int16), np.ascontiguousarray(cr, np.int16)
        if cb.shape != cr.shape:
            raise ValueError('cb and cr must have the same shape')
        self._ck(self._lib.vvcb_chroma_reco_update(self._ctx, _ptr(cb), _ptr(cr), cb.shape[1], x, y, cb.shape[1], cb.shape[0]))

    def chroma_eval(self, visits, want_pred=False):
        """vvcb_chroma_eval: the 8 chroma candidates of every visit (CHROMA_VISIT_DTYPE) with SAD / SATD of Cb and Cr.  Returns the
        CHROMA_RESULT_DTYPE array, or (results, pred) with want_pred: pred is a list of (8, 2, h, w) int16 arrays, one per visit."""
        visits = np.ascontiguousarray(visits, CHROMA_VISIT_DTYPE)
        out = np.zeros(len(visits), CHROMA_RESULT_DTYPE)
        sizes = [2 * CHROMA_CANDS << (int(v['log2w']) + int(v['log2h'])) for v in visits] if want_pred else []
        pred = np.zeros(sum(sizes), np.int16) if want_pred else None
        self._ck(self._lib.vvcb_chroma_eval(self._ctx, _ptr(visits), len(visits), _ptr(pred) if want_pred else None, _ptr(out)))
        if not want_pred:
            return out
        blocks, at = [], 0
        for v, n in zip(visits, sizes):
            blocks.append(pred[at:at + n].reshape(CHROMA_CANDS, 2, 1 << int(v['log2h']), 1 << int(v['log2w'])))
            at += n
        return out, blocks

    def chroma_tu_eval(self, visits, jobs, n_samples, states=None, want_level=False, want_reco=False, want_pred=False):
        """vvcb_chroma_tu_eval: the Cb and Cr TUs of chroma candidates (CHROMA_TU_JOB_DTYPE) of the visits (CHROMA_VISIT_DTYPE).
        states: CHROMA_CTX_STATES_DTYPE array indexed by job['rate_idx'] (needed by DEPQUANT / RATE jobs).  Returns dict with 'results'
        (CHROMA_TU_RESULT_DTYPE) and the wanted flat outputs of n_samples: per candidate Cb w*h, then Cr w*h, at job['offset']."""
        visits = np.ascontiguousarray(visits, CHROMA_VISIT_DTYPE)
        jobs = np.ascontiguousarray(jobs, CHROMA_TU_JOB_DTYPE)
        states = None if states is None else np.ascontiguousarray(states, CHROMA_CTX_STATES_DTYPE)
        out = dict(results=np.zeros(len(jobs), CHROMA_TU_RESULT_DTYPE))
        for key, want, dt in (('level', want_level, np.int32), ('reco', want_reco, np.int16), ('pred', want_pred, np.int16)):
            if want:
                out[key] = np.zeros(n_samples, dt)
        p = lambda k: _ptr(out[k]) if k in out else None
        self._ck(self._lib.vvcb_chroma_tu_eval(self._ctx, _ptr(visits), len(visits), _ptr(jobs), len(jobs),
                                               _ptr(states) if states is not None else None, 0 if states is None else len(states), n_samples,
                                               p('level'), p('reco'), p('pred'), _ptr(out['results'])))
        return out

    def chroma_joint_tu_eval(self, visits, jobs, n_samples, states=None, want_level=False, want_reco=False, want_pred=False):
        """vvcb_chroma_joint_tu_eval: joint Cb-Cr candidates (CHROMA_JOINT_TU_JOB_DTYPE) of the visits (CHROMA_VISIT_DTYPE).
        states: CHROMA_JOINT_CTX_STATES_DTYPE array indexed by job['rate_idx'] (needed by DEPQUANT / RATE jobs).  Returns dict with 'results'
        (CHROMA_JOINT_TU_RESULT_DTYPE) and the wanted flat outputs of n_samples, per candidate 2 w*h at job['offset']: level the coded
        residual's levels then zeros, reco and pred Cb then Cr."""
        visits = np.ascontiguousarray(visits, CHROMA_VISIT_DTYPE)
        jobs = np.ascontiguousarray(jobs, CHROMA_JOINT_TU_JOB_DTYPE)
        states = None if states is None else np.ascontiguousarray(states, CHROMA_JOINT_CTX_STATES_DTYPE)
        out = dict(results=np.zeros(len(jobs), CHROMA_JOINT_TU_RESULT_DTYPE))
        for key, want, dt in (('level', want_level, np.int32), ('reco', want_reco, np.int16), ('pred', want_pred, np.int16)):
            if want:
                out[key] = np.zeros(n_samples, dt)
        p = lambda k: _ptr(out[k]) if k in out else None
        self._ck(self._lib.vvcb_chroma_joint_tu_eval(self._ctx, _ptr(visits), len(visits), _ptr(jobs), len(jobs),
                                                     _ptr(states) if states is not None else None, 0 if states is None else len(states),
                                                     n_samples, p('level'), p('reco'), p('pred'), _ptr(out['results'])))
        return out

    def residual_bits(self, jobs, levels, states):
        """vvcb_residual_bits: fractional bits of residual_coding for the given levels (flat int32 indexed by job['offset'])."""
        jobs = np.ascontiguousarray(jobs, TU_JOB_DTYPE)
        levels = np.ascontiguousarray(levels, np.int32).ravel()
        states = np.ascontiguousarray(states, CTX_STATES_DTYPE)
        bits = np.zeros(len(jobs), np.uint64)
        self._ck(self._lib.vvcb_residual_bits(self._ctx, _ptr(jobs), len(jobs), _ptr(levels), levels.size, _ptr(states), len(states), _ptr(bits)))
        return bits

    @staticmethod
    def calc_rd_cost(lam, frac_bits, distortion):
        """vvcb_calc_rd_cost: RdCost::calcRdCost (pure host logic, no context needed)."""
        return float(load_library().vvcb_calc_rd_cost(float(lam), int(frac_bits), int(distortion)))

    @staticmethod
    def isp_plan(cu_w, cu_h, isp_mode, max_tb_size=64, use_mts=True):
        """vvcb_isp_plan: transform blocks, prediction regions, reference-line lengths and transform types of an intra sub-partition
        CU (CU::canUseISP / getISPSplitDim, getTUIntraSubPartitions, initIntraPatternChTypeISP, TrQuant::getTrTypes).  Pure host logic.
        Returns an ISP_PART_DTYPE array, empty when the CU may not use ISP."""
        parts = np.zeros(4, ISP_PART_DTYPE)
        n = load_library().vvcb_isp_plan(int(cu_w), int(cu_h), int(isp_mode), int(max_tb_size), int(bool(use_mts)), _ptr(parts))
        if n < 0:
            raise EngineError('vvcb_isp_plan: bad argument (sizes are powers of two in 4..64, isp_mode 1 = horizontal or 2 = vertical)')
        return parts[:n]

    @staticmethod
    def isp_mode_param(cu_w, cu_h, pred_w, pred_h, mode):
        """vvcb_isp_mode_param: initPredIntraParams for a prediction region of an ISP CU (pure host logic).  Returns an ISP_MODE_DTYPE record."""
        out = np.zeros(1, ISP_MODE_DTYPE)
        if load_library().vvcb_isp_mode_param(int(cu_w), int(cu_h), int(pred_w), int(pred_h), int(mode), _ptr(out)) != 0:
            raise EngineError('vvcb_isp_mode_param: bad argument')
        return out[0]

    def mts_preselect(self, sums, width, height, max_cand):
        sums = np.ascontiguousarray(sums, np.int32)
        sel = np.zeros(len(sums), np.uint8)
        self._lib.vvcb_mts_preselect(_ptr(sums), len(sums), width, height, max_cand, _ptr(sel))
        return sel

    # ---- texture measures
    def ctu_hads_islice(self, width, height):
        """vvcb_ctu_hads_islice for the frame given to frame_begin (width, height = its luma size)."""
        n = -(-width // self.ctu_size) * -(-height // self.ctu_size)
        out = np.zeros(n, np.int32)
        self._ck(self._lib.vvcb_ctu_hads_islice(self._ctx, _ptr(out), n))
        return out

    def features_eval(self, jobs):
        jobs = np.ascontiguousarray(jobs, FEAT_JOB_DTYPE)
        out = np.zeros(len(jobs), FEAT_RESULT_DTYPE)
        self._ck(self._lib.vvcb_features_eval(self._ctx, _ptr(jobs), len(jobs), _ptr(out)))
        return out

    # ---- device-resident path (bench: kernels without the PCIe copies)
    def dev_alloc(self, nbytes):
        p = C.c_void_p()
        self._ck(self._lib.vvcb_dev_alloc(self._ctx, nbytes, C.byref(p)))
        return p

    def dev_free(self, p):
        self._ck(self._lib.vvcb_dev_free(self._ctx, p))

    def dev_upload(self, dptr, arr):
        arr = np.ascontiguousarray(arr)
        self._ck(self._lib.vvcb_dev_upload(self._ctx, dptr, _ptr(arr), arr.nbytes))

    def dev_download(self, arr, dptr):
        self._ck(self._lib.vvcb_dev_download(self._ctx, _ptr(arr), dptr, arr.nbytes))

    def rmd_eval_device(self, d_visits, n, d_results, d_details=None):
        self._ck(self._lib.vvcb_rmd_eval_device(self._ctx, d_visits, n, d_results, d_details))

    def host_array(self, n, dtype):
        """numpy array of n items backed by page-locked host memory (vvcb_host_alloc).  The memory belongs to the engine: the array (and
        every view of it) must not be used after close()."""
        dtype = np.dtype(dtype)
        p = C.c_void_p()
        nbytes = max(1, n * dtype.itemsize)
        self._ck(self._lib.vvcb_host_alloc(self._ctx, nbytes, C.byref(p)))
        buf = (C.c_char * nbytes).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=n)
        self._pinned = getattr(self, '_pinned', [])
        self._pinned.append(p)
        return arr

    def sync(self):
        self._ck(self._lib.vvcb_sync(self._ctx))

    def timer_start(self):
        self._ck(self._lib.vvcb_timer_start(self._ctx))

    def timer_stop(self):
        ms = C.c_float()
        self._ck(self._lib.vvcb_timer_stop(self._ctx, C.byref(ms)))
        return ms.value

    def measure_int_peak(self):
        """(IMAD-only, IADD3/LOP3-only, mixed) dependent-free issue rates in 1e9 lane-ops/s."""
        a, b, c = C.c_double(), C.c_double(), C.c_double()
        self._ck(self._lib.vvcb_measure_int_peak(self._ctx, C.byref(a), C.byref(b), C.byref(c)))
        return a.value, b.value, c.value

    @property
    def launch_count(self):
        return int(self._lib.vvcb_launch_count(self._ctx))
