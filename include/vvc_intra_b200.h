/*
 * vvc_intra_b200 -- C ABI of the B200 intra cost-evaluation engine.
 *
 * Drop-in boundary for the per-CTU intra cost evaluation behind EncCu::xCompressCU of the VTM 6.1
 * fork llsurreal919/Reduce-Complexity-for-intra-coding-of-VVC.  The reference has no FFI for this
 * path (SURVEY.md 8b); each entry point below names the reference call it replaces.  Abbreviations:
 * EL/ = VVC_project/source/Lib/EncoderLib/, CL/ = VVC_project/source/Lib/CommonLib/.
 *
 * Conventions
 *   - plain pointers and sizes, no C++ types; every function returns VVCB_OK (0) or a negative
 *     error code, vvcb_last_error() gives the text (the reference throws Exception, CL/TypeDef.h:1322;
 *     a host shim turns a non-zero status back into CHECK/THROW).
 *   - sample planes are int16_t (Pel, CL/TypeDef.h:488), row-major, stride in samples (CL/Buffer.h:99).
 *   - all calls are synchronous from the caller's view; one context per host thread / frame in flight.
 *   - there is no CPU fallback: without a CUDA device every call fails with VVCB_ERR_CUDA.
 *   - bit depths 8..10 (the reference's Pel is int16; 11/12 bit would need transform-skip paths that have no golden coverage).
 */
#ifndef VVC_INTRA_B200_H
#define VVC_INTRA_B200_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VVCB_OK            0
#define VVCB_ERR_ARG      -1
#define VVCB_ERR_CUDA     -2
#define VVCB_ERR_STATE    -3

/* ---- evaluation slots of one RMD visit -------------------------------------------------------
 * slot 0..66     regular mode m, reference line 0            (EL/IntraSearch.cpp:489-532, 577-623)
 * slot 67..71    MPM[1..5] on reference line 1               (EL/IntraSearch.cpp:635-681)
 * slot 72..76    MPM[1..5] on reference line 3
 * slot 77..111   MIP mode 0..34                              (EL/IntraSearch.cpp:704-743)          */
#define VVCB_NUM_LUMA_MODE   67
#define VVCB_SLOT_MRL1       67
#define VVCB_SLOT_MRL3       72
#define VVCB_SLOT_MIP        77
#define VVCB_NUM_SLOTS       112
#define VVCB_MAX_LIST        16
#define VVCB_SAT_NONE        0xFFFFFFFFu   /* slot not evaluated for this visit */

/* Fractional-bit prices (SCALE_BITS = 15 fixed point, CL/CommonDef.h:354) of the context-coded bins
 * that xFracModeBitsIntra (EL/IntraSearch.cpp:4263) can touch, read from the CABAC estimator's
 * context snapshot at visit entry (EL/IntraSearch.cpp:301-309).  Bypass bins cost 1<<15.           */
typedef struct vvcb_rates {
  uint32_t mip_flag[2];     /* Ctx::MipFlag(DeriveCtx::CtxMipFlag(cu)), bin 0/1   EL/CABACWriter.cpp:4741 */
  uint32_t mrl_bin0[2];     /* Ctx::MultiRefLineIdx(0)                            EL/CABACWriter.cpp:1566 */
  uint32_t mrl_bin1[2];     /* Ctx::MultiRefLineIdx(1)                                                    */
  uint32_t isp_bin0_0;      /* Ctx::ISPMode(0), bin 0 (ispMode == 0 during RMD)   EL/CABACWriter.cpp:3944 */
  uint32_t mpm_flag[2];     /* Ctx::IntraLumaMpmFlag()                            EL/CABACWriter.cpp:1762 */
  uint32_t planar_flag[2];  /* Ctx::IntraLumaPlanarFlag(1)                                                */
} vvcb_rates;

/* One call of the SATD rough-mode-decision part of IntraSearch::estIntraPredLumaQT
 * (EL/IntraSearch.cpp:430-802) for one luma CU.                                                   */
typedef struct vvcb_rmd_visit {
  int16_t  x, y;              /* luma position in the picture                                          */
  uint8_t  log2w, log2h;      /* 2..6                                                                  */
  /* reference-sample availability in units of 4 samples, as counted by is*Available()
   * (CL/IntraPrediction.cpp:1524-1662): prefix lengths, because constrained intra pred is off.       */
  uint8_t  avail_al;          /* 0/1                                                                   */
  uint8_t  n_above;           /* 0..w/4                                                                */
  uint8_t  n_above_right;     /* 0..w/4                                                                */
  uint8_t  n_left;            /* 0..h/4                                                                */
  uint8_t  n_below_left;      /* 0..h/4                                                                */
  uint8_t  flags;             /* VVCB_VISIT_*                                                          */
  uint8_t  mpm[6];            /* PU::getIntraMPMs (CL/UnitTools.cpp:507)                               */
  uint8_t  num_mpm_cand;      /* its return value (1 or 2): MPMs appended to the RD list (:777-802)    */
  uint8_t  pad[3];
  vvcb_rates rates;
  double   sqrt_lambda;       /* RdCost::getMotionLambda() * FRAC_BITS_SCALE (EL/IntraSearch.cpp:297)  */
} vvcb_rmd_visit;

#define VVCB_VISIT_NO_MRL   1u   /* skip the multi-reference-line pass (derived from y & (ctu-1) if 0)  */
#define VVCB_VISIT_NO_MIP   2u   /* sps.getUseMIP() == false                                            */

typedef struct vvcb_mode {
  uint8_t mip;                /* ModeInfo::mipFlg (EL/IntraSearch.h:190)                               */
  uint8_t mrl;                /* ModeInfo::mRefId: 0, 1 or 3                                           */
  uint8_t mode;               /* ModeInfo::modeId                                                      */
  uint8_t pad;
} vvcb_mode;

#define VVCB_MAX_HAD_LIST   8

/* What the RMD part of estIntraPredLumaQT hands to its full-RD loop (EL/IntraSearch.cpp:1158):        */
typedef struct vvcb_rmd_result {
  int32_t   n_rd, n_had, n_final, pad;
  /* uiRdModeList / CandCostList after the MIP pass and reduceHadCandList (EL/IntraSearch.cpp:747),
   * i.e. what the reference saves at :753-762; costs are IEEE doubles computed in reference order.   */
  vvcb_mode rd_mode[VVCB_MAX_LIST];
  double    rd_cost[VVCB_MAX_LIST];
  /* uiHadModeList / CandHadList (PBINTRA list, :531, :738)                                           */
  vvcb_mode had_mode[VVCB_MAX_HAD_LIST];
  double    had_cost[VVCB_MAX_HAD_LIST];
  /* final full-RD candidate list: rd list + missing MPMs (:777-802)                                  */
  vvcb_mode final_mode[VVCB_MAX_LIST];
} vvcb_rmd_result;

/* Optional per-visit detail (parity, tracing, host-side re-ranking): every evaluated distortion and the
 * regular-only lists as they stood before the MIP pass (what :686-701 saves for blocks < 16x16).      */
typedef struct vvcb_rmd_detail {
  uint32_t  sad [VVCB_NUM_SLOTS];   /* RdCost::xGetSAD  (CL/RdCost.cpp:449);  VVCB_SAT_NONE if skipped  */
  uint32_t  satd[VVCB_NUM_SLOTS];   /* RdCost::xGetHADs (CL/RdCost.cpp:2746)                            */
  int32_t   n_reg, n_reg_had;
  vvcb_mode reg_mode[VVCB_MAX_LIST];
  double    reg_cost[VVCB_MAX_LIST];
  vvcb_mode reg_had_mode[VVCB_MAX_HAD_LIST];
  double    reg_had_cost[VVCB_MAX_HAD_LIST];
} vvcb_rmd_detail;

typedef struct vvcb_ctx vvcb_ctx;

/* ---- life cycle (replaces IntraPrediction::init CL/IntraPrediction.cpp:177, RdCost::init
 *      CL/RdCost.cpp:92, initROM CL/Rom.cpp:263 for this path) ---------------------------------- */
int  vvcb_create (vvcb_ctx** out, int device, int bit_depth, int ctu_size);
void vvcb_destroy(vvcb_ctx* ctx);
const char* vvcb_last_error(const vvcb_ctx* ctx);   /* ctx may be NULL: error of the last failed create */
int  vvcb_device_count(void);
/* Slice-level tool switches the kernels need to know.  VVCB_OPT_DEP_QUANT: slice->getDepQuantEnabledFlag() (default 1, the shipped
 * configuration): residual_coding then picks its significance context set with the quantiser state machine (EL/CABACWriter.cpp:3866). */
#define VVCB_OPT_DEP_QUANT 1
/* VVCB_OPT_YIELD_SYNC (default 0): 1 = the calling thread sleeps while it waits for the device (blocking event) instead of polling; for
 * hosts whose cores are shared with the encoder's walkers (the broker's worker threads).  N in 2..1000 = it looks every N microseconds
 * and sleeps in between (timed sleep instead of the blocking event's interrupt path).                                               */
#define VVCB_OPT_YIELD_SYNC 2
int  vvcb_set_option(vvcb_ctx* ctx, int option, int value);

/* ---- picture planes -------------------------------------------------------------------------
 * frame_begin uploads the (LMCS-mapped) original luma, which is constant during the CTU loop
 * (EL/EncGOP.cpp:1692), and clears the reconstruction plane.  reco_update pushes the rectangle the
 * host has just decided (EncCu::xCompressCU copies the winner into the picture, EL/EncCu.cpp:1581;
 * xRecurIntraCodingLumaQT per tested mode, EL/IntraSearch.cpp:3761).                               */
int vvcb_frame_begin(vvcb_ctx* ctx, const int16_t* orig, int stride, int width, int height);
int vvcb_reco_update(vvcb_ctx* ctx, const int16_t* reco, int stride, int x, int y, int w, int h);

/* reconstruction := original, on the device (no host traffic): the neighbours of the exhaustive candidate sweep (bench.py, configs[4])
 * are taken from the original picture.                                                                              */
int vvcb_reco_from_orig(vvcb_ctx* ctx);

/* Several pictures in one context: vvcb_frame_alloc makes cleared planes of the given size without uploading anything,
 * vvcb_orig_update writes a rectangle of the original plane (what vvcb_reco_update does for the reconstruction).  The broker
 * (vvc_intra_b200_broker.h) keeps the pictures of all its clients side by side in one such plane; a visit's x / y then
 * carry the picture's offset, which must be a multiple of the CTU size.                                             */
int vvcb_frame_alloc(vvcb_ctx* ctx, int width, int height);
/* dst uses the planes of src (same device, src owns them and must outlive dst): several contexts -- one per worker thread of the broker,
 * each with its own stream and scratch -- evaluate requests of different pictures of one plane concurrently.  Rectangle updates through
 * dst write the shared reconstruction plane; callers keep concurrent writers on disjoint pictures.                                    */
int vvcb_frame_share(vvcb_ctx* dst, vvcb_ctx* src);
int vvcb_orig_update(vvcb_ctx* ctx, const int16_t* orig, int stride, int x, int y, int w, int h);
/* Many small reconstruction rectangles in one call (one copy + one scatter kernel): what a host walk pushes before a visit
 * is the few rows above and columns left of the CU (EL/EncCu.cpp:1581, EL/IntraSearch.cpp:3761).  Rectangle i is the dense
 * w*h block at samples + rects[i].offset.                                                                          */
typedef struct vvcb_rect { int16_t x, y, w, h; uint32_t offset; } vvcb_rect;
int vvcb_reco_update_rects(vvcb_ctx* ctx, const vvcb_rect* rects, int n, const int16_t* samples, size_t n_samples);

/* Resident variant: use planes that already live in device memory (from vvcb_dev_alloc); nothing is
 * copied, the caller keeps ownership.  stride in samples, a multiple of 8; both planes 16-byte aligned.
 * Visits evaluated on bound planes through vvcb_rmd_eval_device are NOT validated: they must satisfy what vvcb_rmd_eval checks
 * (sizes 4..64, positions multiples of 4 inside the picture, availability counts within the CU's extent and inside the picture,
 * MPMs < 67); a malformed device-resident visit reads and writes out of bounds.                                                 */
int vvcb_frame_bind_device(vvcb_ctx* ctx, const void* d_orig, const void* d_reco, int stride, int width, int height);

/* ---- rough mode decision: intra prediction + SAD/SATD + mode cost + candidate lists ---------
 * Replaces the RMD block of IntraSearch::estIntraPredLumaQT (EL/IntraSearch.cpp:430-802) for a
 * batch of independent visits: initIntraPatternChType (CL/IntraPrediction.cpp:1064), predIntraAng
 * (:316), initIntraMip/predIntraMip (:2152/:2177), RdCost::xGetSAD/xGetHADs, xFracModeBitsIntra,
 * updateCandList (CL/UnitTools.h:261) and reduceHadCandList (EL/IntraSearch.cpp:4333).
 * visits/results/details are HOST arrays (pinned memory from vvcb_host_alloc makes the copies
 * asynchronous DMA); copies in both directions happen inside the call.                          */
int vvcb_rmd_eval(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_result* results,
                  vvcb_rmd_detail* details /* may be NULL */);

/* The same evaluation with a brief result record (64 bytes instead of 368): what a host walk in an intra slice consumes are the MODES
 * of the lists -- uiRdModeList is the first n_rd entries of the final list (the MPMs of :777-802 are appended behind them) and the
 * Hadamard list's costs only matter to PBINTRA in inter slices (EL/IntraSearch.cpp:966).  A mode code is
 * modeId | mRefId << 8 | mipFlg << 15.  Less than a fifth of the device-to-host traffic of vvcb_rmd_eval.                       */
typedef struct vvcb_rmd_brief {
  uint8_t  n_rd, n_had, n_final, pad;
  uint16_t final_mode[VVCB_MAX_LIST];
  uint16_t had_mode[VVCB_MAX_HAD_LIST];
  uint8_t  reserved[12];
} vvcb_rmd_brief;
int vvcb_rmd_eval_brief(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_brief* out);
/* ... with the visits already resident on the device (uploaded once with vvcb_dev_upload: a static plan such as the exhaustive candidate sweep,
 * the same for every picture): per call only the brief records travel, in chunks that overlap the kernels.  No validation (see
 * vvcb_frame_bind_device).  out: HOST.                                                                                            */
int vvcb_rmd_eval_brief_resident(vvcb_ctx* ctx, const void* d_visits, int n, vvcb_rmd_brief* out);
/* VVCB_OPT_TRUSTED_VISITS (default 0): 1 = the caller guarantees well-formed visits (positions inside the picture, availability
 * within the picture, sizes 4..64): the host-side validation pass of the batch entry points is skipped.                          */
#define VVCB_OPT_TRUSTED_VISITS 3

/* Same work with visits/results already resident on the device (device pointers from
 * vvcb_dev_alloc); used to time the kernels without the PCIe copies.                            */
int vvcb_rmd_eval_device(vvcb_ctx* ctx, const void* d_visits, int n, void* d_results,
                         void* d_details /* may be NULL: no detail tables are written */);

/* Prediction samples of one evaluation slot (debug / parity): writes w*h samples.               */
int vvcb_rmd_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int slot, int16_t* pred);
/* ... of every evaluation slot at once: pred[VVCB_NUM_SLOTS][h][w]; slots the visit does not evaluate are left untouched.  What a
 * host shim at seam S3 (IntraPrediction::predIntraAng / predIntraMip, CL/IntraPrediction.h:176-191) fetches once per visit.        */
int vvcb_rmd_pred_all(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int16_t* pred);

/* ---- TU coding: forward transform, MTS pre-selection sums, scalar quantisation, inverse, reconstruction, SSE ----
 * One job = one candidate transform of one luma TU, i.e. one pass of IntraSearch::xIntraCodingTUBlock
 * (EL/IntraSearch.cpp:2694) after the prediction: TrQuant::transformNxN(trModes) (CL/TrQuant.cpp:1049) when
 * VVCB_TU_QUANT is clear, transformNxN(quant) (:1127) + invTransformNxN (:561) + PelBuf::reconstruct + RdCost::xGetSSE
 * (CL/RdCost.cpp:1739) when it is set.  Quantisation is the scalar Quant::quant (CL/Quant.cpp:994, intra rounding) or,
 * with VVCB_TU_DEPQUANT, the reference's dependent quantisation, or, with VVCB_TU_RDOQ_TS, its RDOQ for transform skip.        */
#define VVCB_TU_QUANT     1u   /* quantise + reconstruct + SSE                                                              */
#define VVCB_TU_DEPQUANT  2u   /* with VVCB_TU_QUANT: dependent (trellis-coded) quantisation, DQIntern::DepQuant::quant
                                  (CL/DepQuant.cpp:1592-1731) and its state-machine dequantiser (:741-810), instead of the
                                  scalar Quant::quant.  Not for transform skip (the reference sends those to RDOQ, :1757).    */
#define VVCB_TU_TS_ALLOWED   8u   /* TU::isTSAllowed  (CL/UnitTools.cpp:4524) -- only read by VVCB_TU_RATE (mts_coding)              */
#define VVCB_TU_MTS_ALLOWED 16u   /* TU::isMTSAllowed (CL/UnitTools.cpp:4549)                                                       */
#define VVCB_TU_RATE        32u   /* with VVCB_TU_QUANT: results[i].frac_bits = fractional bits of CABACWriter::residual_coding( tu, Y ) for
                                     the quantised levels (0 when all levels are zero: the reference does not call it then), priced and
                                     adapted on states[rate_idx]                                                                    */
#define VVCB_TU_RDOQ_TS   4u   /* with VVCB_TU_QUANT, transform skip only: QuantRDOQ::xRateDistOptQuantTS (CL/QuantRDOQ.cpp:1243),
                                  what the shipped configuration (RDOQTS 1) runs for transform-skip candidates; uses lambda and
                                  rate_idx like dependent quantisation.                                                      */

/* Context prices the rate-distortion quantisers read, luma: BinFracBits::intBits[0..1] of each context, taken from the CABAC
 * estimator snapshot the reference passes as `ctx` (ctx.getFracBitsAcess()).  First block: the dependent quantiser's
 * RateEstimator (CL/DepQuant.cpp:479-629).                                                                                 */
typedef struct vvcb_dq_rates {
  uint32_t sig_sbb[2][2];      /* Ctx::SigCoeffGroup[CHANNEL_TYPE_LUMA](0..1)                                                  */
  uint32_t sig[3][12][2];      /* Ctx::SigFlag[0], SigFlag[2], SigFlag[4]: one set per quantiser-state class                   */
  uint32_t par[21][2];         /* Ctx::ParFlag[luma]                                                                          */
  uint32_t gt1[21][2];         /* Ctx::GtxFlag[2 + luma]                                                                      */
  uint32_t gt2[21][2];         /* Ctx::GtxFlag[luma]                                                                          */
  uint32_t last_x[20][2];      /* Ctx::LastX[luma]                                                                            */
  uint32_t last_y[20][2];      /* Ctx::LastY[luma]                                                                            */
  /* transform-skip residual coding, read by QuantRDOQ::xRateDistOptQuantTS (CL/QuantRDOQ.cpp:1243-1485); VVCB_TU_RDOQ_TS only */
  uint32_t ts_sig_sbb[3][2];   /* Ctx::TsSigCoeffGroup                                                                        */
  uint32_t ts_sig[3][2];       /* Ctx::TsSigFlag                                                                              */
  uint32_t ts_par[1][2];       /* Ctx::TsParFlag                                                                              */
  uint32_t ts_gtx[5][2];       /* Ctx::TsGtxFlag                                                                              */
  uint32_t ts_lrg1[4][2];      /* Ctx::TsLrg1Flag                                                                             */
  uint32_t ts_sign[6][2];      /* Ctx::TsResidualSign                                                                         */
} vvcb_dq_rates;

/* Probability states of the CABAC estimator's contexts that CABACWriter::residual_coding touches for a luma TU (EL/CABACWriter.cpp:3773):
 * BinProbModel_Std::m_state[0..1] and m_rate (CL/Contexts.h:90-163) at the moment the reference would start coding the TU.  With
 * VVCB_TU_RATE the engine codes the TU's levels on a private copy of these models exactly as the bit estimator does (every context-coded
 * bin is priced, then adapts its model) and returns the fractional bits.                                                            */
typedef struct vvcb_bin_model { uint16_t state[2]; uint8_t rate; uint8_t pad; } vvcb_bin_model;
typedef struct vvcb_ctx_states {
  vvcb_bin_model mts_idx[11];                                   /* Ctx::MTSIndex                                            */
  vvcb_bin_model sig_sbb[2], sig[3][12], par[21], gt1[21], gt2[21], last_x[20], last_y[20];   /* as vvcb_dq_rates            */
  vvcb_bin_model ts_sig_sbb[3], ts_sig[3], ts_par[1], ts_gtx[5], ts_lrg1[4], ts_sign[6];
} vvcb_ctx_states;

typedef struct vvcb_tu_job {
  int16_t  x, y;            /* luma position of the TU (the original block is read from the frame for the SSE)      */
  uint8_t  log2w, log2h;    /* 2..6; 64-point sides keep their 32 low frequencies (CL/TrQuant.cpp:853)             */
  uint8_t  mts_idx;         /* TransformUnit::mtsIdx: 0 DCT2xDCT2, 1 transform skip, 2..5 DST7/DCT8 pairs (:822-829) */
  uint8_t  flags;           /* VVCB_TU_*                                                                            */
  int16_t  qp_per, qp_rem;  /* QpParam::per / rem of this candidate (CL/Quant.h:71); dependent quantisation adds its +1 itself */
  uint32_t offset;          /* first sample of this job's dense w*h block in resi/pred/coeff/level/reco            */
  /* rate-distortion quantisers (dependent quantisation, transform-skip RDOQ) and LFNST */
  uint16_t rate_idx;        /* which vvcb_dq_rates snapshot prices this TU                                          */
  uint8_t  lfnst_idx;       /* cu.lfnstIdx 0..2: forward LFNST after the primary transform and inverse before it (TrQuant::xFwdLfnst /
                               xInvLfnst, CL/TrQuant.cpp:316-560); the primary transform then keeps the top-left 4x4 / 8x8 only (:853-867)
                               and the dependent quantiser starts at scan position 7 / 15 (CL/DepQuant.cpp:1641-1646)            */
  uint8_t  intra_mode;      /* with lfnst_idx: PU::getFinalIntraMode of the block, PLANAR (0) for MIP (CL/TrQuant.cpp:330-347)        */
  int32_t  cbf_delta_bits;  /* cbfDeltaBits of RateEstimator::xSetLastCoeffOffset (CL/DepQuant.cpp:491-540)          */
  double   lambda;          /* Quant::m_dLambda                                                                     */
} vvcb_tu_job;

typedef struct vvcb_tu_result {
  int32_t  abs_sum_coeff;   /* int(sum |coeff| * scaleSAD), the MTS pre-selection cost (CL/TrQuant.cpp:1090-1103)   */
  int32_t  abs_sum_level;   /* uiAbsSum of the quantiser (0 when VVCB_TU_QUANT is clear)                            */
  uint64_t sse;             /* sum (org - reco)^2 (0 when VVCB_TU_QUANT is clear)                                    */
  uint64_t frac_bits;       /* VVCB_TU_RATE: bits of residual_coding in 1/32768 bit (what getEstFracBits() grows by)  */
} vvcb_tu_result;

/* resi / pred: HOST int16 arrays of n_samples (residual = org - pred as the reference's cs.getResiBuf holds it);
 * coeff / level (int32) and reco (int16): optional HOST outputs of n_samples; results: n entries.                  */
/* rates / states: n_rates entries each (either may be NULL when no job needs it), indexed by job.rate_idx.                      */
int vvcb_tu_eval(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int16_t* resi, const int16_t* pred, size_t n_samples,
                 const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                 int32_t* coeff, int32_t* level, int16_t* reco, vvcb_tu_result* results);
/* The whole of IntraSearch::xIntraCodingTUBlock (EL/IntraSearch.cpp:2694-3168) for TUs that cover their CU: the engine also
 * runs initIntraPatternChType + predIntraAng / predIntraMip (:2820-2870) from the reconstruction plane and forms
 * resi = org - pred (:2922) itself.  src[i] names the visit (position, size, availability: the same struct the rough mode
 * decision takes) and the evaluation slot (VVCB_SLOT_*) of job i; jobs[i] must have the visit's position and size.
 * pred_out (optional, HOST, n_samples): the prediction samples.                                                        */
typedef struct vvcb_tu_src {
  uint32_t visit;           /* index into visits[]                                                                  */
  uint8_t  slot;            /* evaluation slot: regular mode, MPM on reference line 1 / 3, or MIP mode              */
  uint8_t  pad[3];
} vvcb_tu_src;
int vvcb_tu_eval_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_tu_src* src, const vvcb_tu_job* jobs, int n,
                      size_t n_samples, const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                      int32_t* coeff, int32_t* level, int16_t* reco, int16_t* pred_out, vvcb_tu_result* results);
/* ---- one round trip per CU of the host walk ----------------------------------------------------------------------------
 * What IntraSearch::estIntraPredLumaQT (EL/IntraSearch.cpp:289) needs from the engine for one luma CU, in one call: push the
 * reconstructed neighbourhood (rects), run the rough mode decision of the visit (want_rmd: lists + every SAD / SATD, :430-802) and
 * code a set of candidate TUs of that CU (jobs: xIntraCodingTUBlock, :2694, for the (mode, transform, LFNST) combinations the
 * full-RD loop :1158 may reach; all priced on one context snapshot, rate_idx 0, because the reference restores the estimator
 * before every candidate, :1222 / :3448).  slots[k] is the evaluation slot (VVCB_SLOT_*) of job k; jobs[k].offset addresses this
 * request's own level / reco / pred arrays (n_jobs dense w*h blocks).  The requests of one call are independent: they may
 * belong to different pictures of the plane (broker), which is why the reconstruction rectangles travel with them.            */
/* Candidates named by the engine itself: which modes survive the rough mode decision is only known after it ran, so a request may carry
 * TEMPLATES instead of jobs -- (transform, LFNST index, flags, QP, lambda) prototypes -- and the engine combines each with every mode of
 * the visit's final list (modes & VVCB_AUTO_FINAL) and / or of the regular-only list of vvcb_rmd_detail that is not in the final list
 * (modes & VVCB_AUTO_REGULAR: what the LFNST passes of small blocks restore, EL/IntraSearch.cpp:686-701), modes in list order, templates in
 * the given order; skip_mip drops MIP modes (LFNST is not combined with MIP for small blocks, allowLfnstWithMip).  One round trip instead of two. */
#define VVCB_AUTO_FINAL    1u
#define VVCB_AUTO_REGULAR  2u
typedef struct vvcb_cu_auto {
  vvcb_tu_job job;            /* prototype: position, size, mts_idx, flags, QP, lfnst_idx, lambda, cbf_delta_bits; offset / intra_mode / rate_idx are filled in */
  uint8_t modes;              /* VVCB_AUTO_*                                                                                       */
  uint8_t skip_mip;
  uint8_t pad[6];
} vvcb_cu_auto;

typedef struct vvcb_cu_request {
  const vvcb_rect* rects; int n_rects; const int16_t* rect_samples; size_t n_rect_samples;
  const vvcb_rmd_visit* visit;           /* may be NULL when the request only pushes rectangles                                  */
  int want_rmd;
  const vvcb_tu_job* jobs; const uint8_t* slots; int n_jobs;
  const vvcb_dq_rates* rates; const vvcb_ctx_states* states;   /* one snapshot each (NULL when no job needs it)                  */
  vvcb_rmd_result* result; vvcb_rmd_detail* detail;            /* outputs of want_rmd (detail optional)                          */
  int32_t* level; int16_t* reco; int16_t* pred;                /* optional outputs of the jobs, n_jobs * w * h each              */
  vvcb_tu_result* tu_results;                                  /* n_jobs                                                         */
  /* templates (need want_rmd, and detail when a template names the regular-only list); the expanded candidates come back in the auto_* arrays */
  const vvcb_cu_auto* autos; int n_autos; int max_auto;        /* max_auto: capacity of the auto_* arrays (further candidates are dropped) */
  int* n_auto;                                                 /* out: number of expanded candidates                             */
  uint8_t* auto_slot; uint8_t* auto_tmpl;                      /* out: evaluation slot and template index of each                */
  int32_t* auto_level; int16_t* auto_reco; int16_t* auto_pred; /* optional outputs, max_auto * w * h each                        */
  vvcb_tu_result* auto_results;                                /* max_auto                                                       */
} vvcb_cu_request;
int vvcb_cu_eval(vvcb_ctx* ctx, vvcb_cu_request* reqs, int n);

/* The residual part of IntraSearch::xGetIntraFracBitsQT (EL/IntraSearch.cpp:2566: xEncCoeffQT -> CABACWriter::residual_coding on the bit
 * estimator) for levels the caller already has.  levels: HOST int32, dense w*h per job at job.offset; of a job only log2w, log2h, mts_idx,
 * the VVCB_TU_TS_ALLOWED / VVCB_TU_MTS_ALLOWED flags, offset and rate_idx are read; bits[i]: fractional bits, 0 for an all-zero block.      */
int vvcb_residual_bits(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int32_t* levels, size_t n_samples,
                       const vvcb_ctx_states* states, int n_states, uint64_t* bits);
/* TrQuant::transformNxN(trModes) candidate selection (CL/TrQuant.cpp:1112-1123) from the pre-selection sums of one
 * TU's candidates in list order (DCT2 first, transform skip second if tested): pure host logic.                    */
void vvcb_mts_preselect(const int32_t* sums, int n, int width, int height, int max_cand, uint8_t* selected);
/* RdCost::calcRdCost (CL/RdCost.cpp:63-74): (32768 / lambda) * distortion + frac_bits in IEEE double, the reference's operation order
 * (lambda = RdCost::getLambda()).  Pure host logic: cost of a candidate from vvcb_tu_result::sse and the bits the walk has summed
 * (vvcb_tu_result::frac_bits + its own header bits).                                                                          */
double vvcb_calc_rd_cost(double lambda, uint64_t frac_bits, uint64_t distortion);

/* ---- intra sub-partitions (ISP): geometry of one luma CU (pure host logic; SURVEY 8 row f1, first slice) ----------------------------
 * What the job builder of an ISP candidate needs before any kernel runs, as the reference derives it:
 *   CU::canUseISP (CL/UnitTools.cpp:426)  -- log2w + log2h > 4 and neither side above max_tb_size;
 *   CU::getISPSplitDim (:437) and PartitionerImpl::getTUIntraSubPartitions (CL/UnitPartitioner.cpp:978) -- 2 or 4 transform blocks,
 *     each of at least 16 samples, stacked along the split direction;
 *   CU::isPredRegDiffFromTB / isFirstTBInPredReg / adjustPredArea (CL/UnitTools.cpp:4334-4355) -- vertical split of a 4xN or 8xN (N > 4)
 *     CU: the 1xN / 2xN transform blocks are predicted in regions 4 samples wide, at the first block of each region;
 *   IntraPrediction::initIntraPatternChTypeISP (CL/IntraPrediction.cpp:1092-1203) -- reference-line lengths: the first region fetches
 *     the lines of the whole CU once (fetch_*), every region then predicts with top = cu_w + pred_w, left = cu_h + pred_h samples;
 *   TrQuant::getTrTypes (CL/TrQuant.cpp:752-783) -- ISP blocks take DST-VII in a direction of 4..16 samples, DCT-II otherwise
 *     (DCT-II in both when the SPS switches MTS off: use_mts = sps.getUseMTS()).
 * vvcb_isp_eval (below) evaluates ISP candidates whose transform blocks are all at least 4x4 (horizontal split: CU height >= 16 or the
 * 4x8 CU; vertical split: CU width >= 16 or the 8x4 CU).  NOT in the library yet: the 1xN / 2xN / Nx1 / Nx2 blocks (one-dimensional and
 * 2-point transforms, their scans and contexts, the 4-wide prediction rule) and LFNST with ISP; the served encoder still hands ISP
 * candidates to the reference code (DESIGN.md 7).                                                                                      */
#define VVCB_ISP_NONE 0
#define VVCB_ISP_HOR  1   /* HOR_INTRA_SUBPARTITIONS: blocks stacked top to bottom (TU_1D_HORZ_SPLIT) */
#define VVCB_ISP_VER  2   /* VER_INTRA_SUBPARTITIONS: blocks side by side (TU_1D_VERT_SPLIT)          */
#define VVCB_TR_DCT2  0   /* TransType (CL/TypeDef.h) */
#define VVCB_TR_DCT8  1
#define VVCB_TR_DST7  2
#define VVCB_ISP_MAX_PARTS 4
typedef struct vvcb_isp_part {
  int16_t x, y, w, h;                      /* transform block, luma samples relative to the CU's top-left                          */
  int16_t pred_x, pred_y, pred_w, pred_h;  /* prediction region the block lies in (== the block unless the 4-wide rule applies)     */
  int16_t top_ref_len, left_ref_len;       /* m_topRefLength / m_leftRefLength while this region is predicted                       */
  int16_t fetch_top_len, fetch_left_len;   /* first block only: lengths of the one xFillReferenceSamples over the CU; else 0        */
  uint8_t predicts;                        /* 1: the region's prediction is made when this block is coded (isFirstTBInPredReg)      */
  uint8_t tr_hor, tr_ver;                  /* VVCB_TR_*                                                                             */
  uint8_t last;                            /* CU::isISPLast                                                                         */
} vvcb_isp_part;                           /* 28 bytes */
/* parts: room for VVCB_ISP_MAX_PARTS.  Returns the number of blocks (2 or 4), 0 when the CU may not use ISP (canUseISP false),
 * VVCB_ERR_ARG for sizes that are not powers of two in 4..64, an isp_mode other than VVCB_ISP_HOR / VVCB_ISP_VER, or parts == NULL. */
int vvcb_isp_plan(int cu_w, int cu_h, int isp_mode, int max_tb_size, int use_mts, vvcb_isp_part* parts);
/* IntraPrediction::initPredIntraParams (CL/IntraPrediction.cpp:487-618) for a prediction region (vvcb_isp_part::pred_w x pred_h) of an ISP CU and
 * one luma mode 0..66: the wide-angle remap takes the CU's shape, PDPC (regions of at least 4x4 only) and its scale the region's; the reference
 * lines are never smoothed and the interpolation is the cubic one (refFilterFlag = interpolationFlag = false), reference line 0.               */
typedef struct vvcb_isp_mode {
  int16_t  angle;       /* intraPredAngle, 0 for planar / DC                       */
  uint16_t inv_angle;   /* invAngle                                                */
  uint8_t  is_ver;      /* isModeVer (after the wide-angle remap)                  */
  uint8_t  pdpc;        /* applyPDPC                                               */
  int8_t   ang_scale;   /* angularScale, meaningful for positive angles with pdpc  */
  uint8_t  pad;
} vvcb_isp_mode;        /* 8 bytes */
int vvcb_isp_mode_param(int cu_w, int cu_h, int pred_w, int pred_h, int mode, vvcb_isp_mode* out);

/* Evaluation of ISP candidates: the luma part of IntraSearch::xIntraCodingLumaISP (EL/IntraSearch.cpp:3171) for CUs whose blocks are at
 * least 4x4.  A candidate is one CU x split x luma mode x quantiser setting; its blocks are coded in order on one estimator, as the
 * reference does after restoring the CABAC estimator once per candidate: initIntraPatternChTypeISP + predIntraAng of block k from the
 * reconstruction of block k-1 (CL/IntraPrediction.cpp:1092-1203; lines unfiltered, cubic interpolation, reference line 0),
 * TrQuant::transformNxN with the implicit DST-VII / DCT-II pair (CL/TrQuant.cpp:752-783), Quant::quant or DepQuant::quant with
 * cbfDeltaBits of the ISP branch of RateEstimator::xSetLastCoeffOffset (CL/DepQuant.cpp:491-540), invTransformNxN, reconstruction and SSE
 * (xIntraCodingTUBlock, :2694), then xGetIntraFracBitsQT's cbf bin (Ctx::QtCbf[luma](2 + cbf of the previous block); the last block's cbf
 * is not coded when every earlier one is 0) and residual_coding, each block priced on the context models the previous block left.
 * Header bits (mode, ISP flag, LFNST index) stay with the caller, and so do the early exits of the reference's loop (bestCostSoFar): they
 * never change the value of a block that is computed, so every block is computed and the per-block results let the caller apply them.
 * Blocks of 1 or 2 samples in one direction, LFNST, transform skip and explicit MTS are not evaluated (vvcb_isp_plan describes them).    */
typedef struct vvcb_isp_job {
  uint32_t visit;            /* index into visits[]: the CU (position, size, availability); mpm / rates / sqrt_lambda are not read      */
  uint8_t  isp_mode;         /* VVCB_ISP_HOR / VVCB_ISP_VER                                                                          */
  uint8_t  mode;             /* luma mode 0..66                                                                                      */
  uint8_t  flags;            /* VVCB_TU_QUANT [| VVCB_TU_DEPQUANT] [| VVCB_TU_RATE]                                                  */
  uint8_t  use_mts;          /* sps.getUseMTS(): DST-VII for block sides 4..16                                                       */
  uint8_t  max_tb_size;      /* sps max TB size (CU::canUseISP)                                                                      */
  uint8_t  lfnst_idx;        /* must be 0                                                                                            */
  int16_t  qp_per, qp_rem;   /* as vvcb_tu_job                                                                                       */
  uint16_t rate_idx;         /* states[rate_idx]: the estimator's models at the start of the candidate                               */
  uint32_t offset;           /* first sample of this candidate's cu_w*cu_h outputs: its blocks in coding order, each dense w*h      */
  vvcb_bin_model cbf[2];     /* Ctx::QtCbf[luma] contexts 2 and 3 at the start of the candidate                                      */
  double   lambda;           /* Quant::m_dLambda (dependent quantisation)                                                            */
} vvcb_isp_job;              /* 40 bytes */
typedef struct vvcb_isp_result {
  vvcb_tu_result part[VVCB_ISP_MAX_PARTS];  /* per block, coding order: abs sums, sse, residual frac_bits (VVCB_TU_RATE)             */
  uint32_t cbf_bits[VVCB_ISP_MAX_PARTS];    /* fractional bits of the block's cbf bin, 0 when it is inferred                        */
  uint8_t  cbf[VVCB_ISP_MAX_PARTS];
  uint8_t  n_parts;                         /* 2 or 4                                                                               */
  uint8_t  discarded;                       /* the last cbf is inferred but the last block has no level: the reference gives the
                                               candidate MAX_INT distortion                                                          */
  uint8_t  pad[2];
} vvcb_isp_result;                          /* 120 bytes */
/* visits: HOST, the CUs (availability must be all or nothing on each side: n_left 0 or h/4, n_above 0 or w/4, and no below-left /
 * above-right without it -- in a tree partition the left and above of a CU's own rows and columns are coded before it, and only then
 * does the fresh fetch of the device agree with the reference's shifted lines).  level / reco / pred: optional HOST outputs of n_samples.
 * Needs vvcb_frame_begin (original and reconstruction planes).  Returns VVCB_ERR_ARG for a CU or split without blocks of at least 4x4,
 * other availability, mode > 66, lfnst_idx != 0, transform-skip / RDOQ flags, a bad rate_idx, lambda <= 0 with VVCB_TU_DEPQUANT, or
 * outputs outside n_samples.                                                                                                       */
int vvcb_isp_eval(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_isp_job* jobs, int n,
                  const vvcb_ctx_states* states, int n_states, size_t n_samples,
                  int32_t* level, int16_t* reco, int16_t* pred, vvcb_isp_result* results);

/* ---- chroma intra candidates (4:2:0, separate tree): prediction + SAD / SATD of Cb and Cr ------------------------------------------
 * The data-parallel half of IntraSearch::estIntraPredChromaQT (EL/IntraSearch.cpp:1382), which every chroma CU of the separate tree of an
 * all-intra picture runs (EL/EncCu.cpp:519-536): the candidates of PU::getIntraChromaCandModes (CL/UnitTools.cpp) predicted for Cb and
 * Cr -- planar / DC / angular with the chroma rules of initPredIntraParams and xPredIntraAng (CL/IntraPrediction.cpp:487-618, 633-935:
 * parameters from the chroma block's own shape, reference lines never smoothed, the 2-tap linear interpolation) and the cross-component
 * modes (CL/IntraPrediction.cpp:1665-2150: xGetLumaRecPixels with the [1 2 1; 1 2 1] / 8 down-sampling of sps_cclm_colocated_chroma
 * = 0, xGetLMParameters, predIntraChromaLM) -- and measured with RdCost::xGetSAD / xGetHADs on the chroma block.  No ordering or
 * pruning of the candidates: that is the caller's.  vvcb_chroma_tu_eval (below) codes the TUs of these candidates, Cb and Cr
 * separately with DCT-II, and vvcb_chroma_joint_tu_eval their joint Cb-Cr tries; chroma transform skip and the chroma QP mapping are
 * not in the library.
 * Restated from H.266 and the cited reference lines; not compared with the reference encoder's own chroma output.                   */
#define VVCB_CHROMA_CANDS 8
#define VVCB_LM_CHROMA   67   /* LM_CHROMA_IDX: CCLM from the above and left neighbours */
#define VVCB_MDLM_L      68   /* MDLM_L_IDX: left and below-left only                    */
#define VVCB_MDLM_T      69   /* MDLM_T_IDX: above and above-right only                  */
#define VVCB_DM_CHROMA   70   /* DM_CHROMA_IDX: the derived luma mode (vvcb_chroma_visit::dm_mode) */

/* Chroma planes of the picture given to vvcb_frame_begin: Cb / Cr originals, their reconstructions cleared.  cw = width / 2,
 * ch = height / 2 (4:2:0); bit depth = the context's.  The CCLM modes read the context's luma reconstruction (vvcb_reco_update /
 * vvcb_reco_update_rects): in the separate tree the whole luma CTU is coded before its chroma.                                   */
int vvcb_chroma_frame_begin(vvcb_ctx* ctx, const int16_t* cb, const int16_t* cr, int stride, int cw, int ch);
/* the rectangle (chroma samples) of both reconstructions the host has just decided */
int vvcb_chroma_reco_update(vvcb_ctx* ctx, const int16_t* cb, const int16_t* cr, int stride, int x, int y, int w, int h);

/* One chroma CU of the separate tree. */
typedef struct vvcb_chroma_visit {
  int16_t x, y;              /* chroma position, even                                                                           */
  uint8_t log2w, log2h;      /* 2..5 (2xN / Nx2 are not evaluated)                                                              */
  /* reference-sample availability in the reference's chroma units of 2 samples (pcv.minCUWidth >> scaleX), prefix counts as for
   * vvcb_rmd_visit: avail_al 0/1, n_above / n_above_right 0..w/2, n_left / n_below_left 0..h/2.  CCLM takes a side only when it is
   * whole (n_above == w/2, n_left == h/2), and the above-right / below-left only with their side.                                   */
  uint8_t avail_al, n_above, n_above_right, n_left, n_below_left;
  uint8_t dm_mode;           /* the derived luma mode 0..66 (PLANAR when the collocated luma CU is MIP), kept by the caller's walk */
  uint8_t cclm;              /* 1: the LM modes are evaluated (PU::isLMCModeEnabled, the caller's decision)                        */
  uint8_t pad[3];
} vvcb_chroma_visit;         /* 16 bytes */

/* The 8 candidates in the reference's order: PLANAR, VER (50), HOR (18), DC, LM, MDLM_L, MDLM_T, DM; the first of the four regular ones
 * that equals dm_mode is VDIA (66) instead.  sad / satd [candidate][0 Cb, 1 Cr]; VVCB_SAT_NONE: not evaluated (LM modes without cclm). */
typedef struct vvcb_chroma_result {
  uint8_t  mode[VVCB_CHROMA_CANDS];        /* 0..66, VVCB_LM_CHROMA / VVCB_MDLM_L / VVCB_MDLM_T, VVCB_DM_CHROMA (predicts dm_mode) */
  uint32_t sad[VVCB_CHROMA_CANDS][2];
  uint32_t satd[VVCB_CHROMA_CANDS][2];
} vvcb_chroma_result;        /* 136 bytes */

/* visits / results: HOST arrays of n.  pred_out (optional, HOST): per visit, in order, 8 x 2 x w*h int16 -- [candidate][Cb, Cr][h][w]
 * (the blocks of LM candidates that are not evaluated are zero).  VVCB_ERR_ARG for sides outside 4..32, odd positions,
 * counts above their maximum, dm_mode > 66, a CU or neighbour outside the chroma picture; VVCB_ERR_STATE before
 * vvcb_chroma_frame_begin and through the broker.                                                                                 */
int vvcb_chroma_eval(vvcb_ctx* ctx, const vvcb_chroma_visit* visits, int n, int16_t* pred_out, vvcb_chroma_result* results);

/* ---- chroma TU coding of the candidates (4:2:0, separate tree, Cb and Cr coded separately) -------------------------------------
 * The chroma part of IntraSearch::xRecurIntraChromaCodingQT (EL/IntraSearch.cpp) for a TU that covers its chroma CU -- xIntraCodingTUBlock
 * (:2694) of Cb, then of Cr -- and the chroma bins of xGetIntraFracBitsQT (:2566), for the candidates estIntraPredChromaQT prices on their
 * full RD cost.  A job is one chroma CU (visit), one of its 8 candidates and one quantiser setting:
 *   - prediction: exactly what vvcb_chroma_eval predicts for (visit, cand), the LM modes from the context's luma reconstruction;
 *     residual = original - prediction, from the planes of vvcb_chroma_frame_begin;
 *   - TrQuant::transformNxN with DCT-II in both directions, Quant::quant (scalar, intra rounding) or, with VVCB_TU_DEPQUANT,
 *     DepQuant::quant on the chroma context sets and per-position offsets of H.266 9.3.4.2.5-9.3.4.2.8: significance context
 *     36 + 8 * max(0, state - 1) + min((sumAbs1 + 1) >> 1, 3) + (d < 2 ? 4 : 0), greater-than / parity context
 *     min(sumAbs1 - numPos, 4) + 1 + (d == 0 ? 5 : 0) (d = x + y), last-position prefix contexts from offset 20 with shift
 *     Clip3(0, 2, side >> 3), coded-sub-block flag contexts 2..3; then the dequantiser, invTransformNxN, reconstruction and RdCost::xGetSSE;
 *   - cbfDeltaBits (RateEstimator::xSetLastCoeffOffset, CL/DepQuant.cpp:491-540): Cb's from Ctx::QtCbf[Cb](0), Cr's from Ctx::QtCbf[Cr]
 *     selected by Cb's final cbf (prevCbf); so Cr is quantised after Cb's levels are final.  Both quantisers are priced on the
 *     candidate's starting snapshot states[rate_idx];
 *   - with VVCB_TU_RATE: the chroma bins of transform_unit on ONE carried copy of states[rate_idx], in coding order -- tu_cb_coded_flag
 *     (context 0), tu_cr_coded_flag (context = Cb's cbf), residual_coding of Cb, residual_coding of Cr (priced on the models Cb's
 *     residual left); each bin priced, then its model adapted.  Sign hiding is not modelled (as for luma).
 * Restated from H.266 and the cited reference lines, as the ISP and chroma-prediction entries are: parity with the reference encoder's
 * own chroma coding is unpinned.  Joint Cb-Cr candidates are coded by vvcb_chroma_joint_tu_eval (below).  NOT in the library: chroma
 * transform skip (its transform_skip_flag bin has contexts of its own and stays with the caller), LFNST for chroma, the chroma QP mapping (the caller passes QpParam per component, its mapping
 * table and offsets applied), chroma distortion weighting (the caller applies m_distortionWeight to sse), 2xN blocks, 4:2:2 / 4:4:4,
 * ISP-coupled chroma.                                                                                                              */
typedef struct vvcb_chroma_ctx_states {   /* the estimator's chroma models at the start of the chroma TU (as vvcb_ctx_states)       */
  vvcb_bin_model cbf_cb[2], cbf_cr[3];   /* Ctx::QtCbf[Cb] / [Cr] (tu_cb_coded_flag: 2 contexts, tu_cr_coded_flag: 3)           */
  vvcb_bin_model sig_sbb[2];             /* Ctx::SigCoeffGroup[CHANNEL_TYPE_CHROMA]                                              */
  vvcb_bin_model sig[3][8];              /* Ctx::SigFlag[1], [3], [5]: one set per quantiser-state class                          */
  vvcb_bin_model par[11], gt1[11], gt2[11];   /* Ctx::ParFlag[chroma], GtxFlag[3], GtxFlag[1]                                   */
  vvcb_bin_model last_x[3], last_y[3];   /* Ctx::LastX / LastY[chroma]                                                           */
} vvcb_chroma_ctx_states;                /* 70 models, 420 bytes */
typedef struct vvcb_chroma_tu_job {
  uint32_t visit;              /* index into visits[]                                                                            */
  uint8_t  cand;               /* 0..7, the candidate order of vvcb_chroma_result, the DM -> VDIA substitution included          */
  uint8_t  flags;              /* VVCB_TU_QUANT [| VVCB_TU_DEPQUANT] [| VVCB_TU_RATE]                                            */
  uint16_t rate_idx;           /* states[rate_idx]: the models at the start of the candidate (DEPQUANT or RATE)                  */
  int16_t  qp_per[2], qp_rem[2];   /* QpParam(tu, COMPONENT_Cb / Cr): the caller's chroma QP mapping and offsets applied          */
  uint32_t offset;             /* first sample of this candidate's outputs: Cb w*h, then Cr w*h                                  */
  uint32_t pad;
  double   lambda[2];          /* Quant::m_dLambda while Cb / Cr are quantised (DEPQUANT)                                        */
} vvcb_chroma_tu_job;          /* 40 bytes */
typedef struct vvcb_chroma_tu_result {
  vvcb_tu_result comp[2];      /* Cb, Cr: abs sums, unweighted sse (xGetSSE), residual frac_bits (VVCB_TU_RATE, 0 without a level) */
  uint32_t cbf_bits[2];        /* VVCB_TU_RATE: fractional bits of tu_cb_coded_flag / tu_cr_coded_flag                           */
  uint8_t  cbf[2], pad[6];
} vvcb_chroma_tu_result;       /* 64 bytes */
/* visits, jobs, states: HOST arrays (n_visits, n, n_states; states may be NULL when no job has DEPQUANT or RATE).  level / reco / pred:
 * optional HOST outputs of n_samples.  VVCB_ERR_ARG for a visit vvcb_chroma_eval refuses, cand > 7, an LM candidate of a visit with
 * cclm == 0, other flags, per / rem out of range for the bit depth, a bad rate_idx, lambda <= 0 with DEPQUANT, or outputs outside
 * n_samples; VVCB_ERR_STATE before vvcb_chroma_frame_begin and through the broker.                                                 */
int vvcb_chroma_tu_eval(vvcb_ctx* ctx, const vvcb_chroma_visit* visits, int n_visits, const vvcb_chroma_tu_job* jobs, int n,
                        const vvcb_chroma_ctx_states* states, int n_states, size_t n_samples,
                        int32_t* level, int16_t* reco, int16_t* pred, vvcb_chroma_tu_result* results);

/* ---- joint Cb-Cr coding of the candidates (4:2:0, separate tree, one coded residual for both components) -----------------------
 * The joint Cb-Cr tries of xRecurIntraChromaCodingQT for a TU that covers its chroma CU: one residual stands for Cb and Cr under
 * TuCResMode `mode` (H.266 7.4.11.10, 8.7.2) -- 1: tu_cb_coded_flag 1, tu_cr_coded_flag 0; 2: both 1; 3: tu_cb_coded_flag 0,
 * tu_cr_coded_flag 1 -- and CSign = `sign` = 1 - 2 * slice_joint_cbcr_sign_flag.  A job is one chroma CU, one of its 8 candidates,
 * mode, sign and one quantiser setting (one QP, one lambda):
 *   - prediction of Cb and Cr: exactly what vvcb_chroma_eval predicts for (visit, cand); resCb / resCr = original - prediction;
 *   - forward combination into the coded residual.  H.266 does not specify it; this is the library's restatement of the encoder
 *     derivation of JVET-O0105 (C division, truncating toward zero), and parity with the reference encoder's own is unpinned:
 *     mode 2: (resCb + CSign * resCr) / 2;  mode 1: (4 * resCb + 2 * CSign * resCr) / 5;  mode 3: (4 * resCr + 2 * CSign * resCb) / 5.
 *     It decides only which levels are chosen, never whether the reconstruction of given levels is right;
 *   - DCT-II, Quant::quant or DepQuant::quant on the chroma contexts, dequantiser and inverse transform of that one residual, as
 *     vvcb_chroma_tu_eval codes Cb.  cbfDeltaBits belong to the coded component (the reading of RateEstimator::xSetLastCoeffOffset
 *     cited above): Ctx::QtCbf[Cb](0) for modes 1 and 2, Ctx::QtCbf[Cr](0) for mode 3, where tu_cb_coded_flag is 0;
 *   - inverse mapping (normative, H.266 8.7.2), in int, with r the inverse-transformed residual after its 16-bit clip:
 *     mode 1: resCb = r, resCr = (CSign * r) >> 1;  mode 2: resCb = r, resCr = CSign * r;  mode 3: resCr = r, resCb = (CSign * r) >> 1;
 *     then Clip1(prediction + residual) of both components and their unweighted RdCost::xGetSSE;
 *   - with VVCB_TU_RATE: the chroma bins of transform_unit in coding order on ONE carried copy of states[rate_idx], each priced, then
 *     adapted -- tu_cb_coded_flag (context 0), tu_cr_coded_flag (context = tu_cb_coded_flag), tu_joint_cbcr_residual_flag = 1
 *     (context 2 * tu_cb_coded_flag + tu_cr_coded_flag - 1), residual_coding of the coded residual on the chroma contexts.
 * A coded residual whose levels are all zero is not a joint candidate (the syntax cannot code it): cbf = 0, the reconstruction and sse of
 * the zero residual, no bins priced; the caller discards it.  The chroma QP mapping with the joint QP offsets, the distortion weights
 * and the choice of modes and slice sign stay with the caller.  Restated from H.266 and the cited lines; parity unpinned.          */
typedef struct vvcb_chroma_joint_ctx_states {
  vvcb_chroma_ctx_states chroma;         /* the models of vvcb_chroma_tu_eval                                                      */
  vvcb_bin_model joint[3];               /* Ctx::JointCbCrFlag                                                                     */
} vvcb_chroma_joint_ctx_states;          /* 73 models, 438 bytes */
typedef struct vvcb_chroma_joint_tu_job {
  uint32_t visit;              /* index into visits[]                                                                            */
  uint8_t  cand;               /* 0..7, as vvcb_chroma_tu_job::cand                                                              */
  uint8_t  flags;              /* VVCB_TU_QUANT [| VVCB_TU_DEPQUANT] [| VVCB_TU_RATE]                                            */
  uint16_t rate_idx;           /* states[rate_idx]: the models at the start of the candidate (DEPQUANT or RATE)                  */
  uint8_t  mode;               /* TuCResMode 1..3                                                                                */
  int8_t   sign;               /* CSign: +1 or -1                                                                                */
  int16_t  qp_per, qp_rem;     /* QpParam of the joint residual: the caller's chroma QP mapping and joint offsets applied        */
  uint16_t pad;
  uint32_t offset;             /* first sample of this candidate's outputs: Cb w*h, then Cr w*h                                  */
  uint32_t pad2;
  double   lambda;             /* Quant::m_dLambda while the joint residual is quantised (DEPQUANT)                              */
} vvcb_chroma_joint_tu_job;    /* 32 bytes */
typedef struct vvcb_chroma_joint_tu_result {
  vvcb_tu_result res;          /* the coded residual: abs sums, residual frac_bits (VVCB_TU_RATE, 0 without a level); sse unused (0) */
  uint64_t sse[2];             /* Cb, Cr: unweighted sse of the reconstructions                                                  */
  uint32_t cbf_bits[2];        /* VVCB_TU_RATE: fractional bits of tu_cb_coded_flag / tu_cr_coded_flag                           */
  uint32_t joint_bits;         /* VVCB_TU_RATE: fractional bits of tu_joint_cbcr_residual_flag                                   */
  uint8_t  cbf, pad[3];        /* 1: the coded residual has a level; 0: not a joint candidate                                    */
} vvcb_chroma_joint_tu_result; /* 56 bytes */
/* visits, jobs, states: HOST arrays (n_visits, n, n_states; states may be NULL when no job has DEPQUANT or RATE).  level / reco / pred:
 * optional HOST outputs of n_samples, per candidate 2 * w*h at its offset: level the coded residual's levels, then w*h zeros; reco and
 * pred Cb, then Cr.  VVCB_ERR_ARG for everything vvcb_chroma_tu_eval refuses and for mode outside 1..3 or sign other than +1 / -1;
 * VVCB_ERR_STATE before vvcb_chroma_frame_begin and through the broker.                                                            */
int vvcb_chroma_joint_tu_eval(vvcb_ctx* ctx, const vvcb_chroma_visit* visits, int n_visits, const vvcb_chroma_joint_tu_job* jobs, int n,
                              const vvcb_chroma_joint_ctx_states* states, int n_states, size_t n_samples,
                              int32_t* level, int16_t* reco, int16_t* pred, vvcb_chroma_joint_tu_result* results);

/* ---- texture features (orig-only, trivially parallel) ------------------------------------------------------------
 * vvcb_ctu_hads_islice: EncCu::updateCtuDataISlice (EL/EncCu.cpp:564-675) for every CTU of the frame, as
 * EncSlice::calCostSliceI calls it (EL/EncSlice.cpp:1276-1298): sum over the complete 8x8 blocks of the CTU's
 * original luma of (Hadamard AC sum + 2) >> 2.  out[ctuRsAddr], n_ctus = ceil(w/ctu)*ceil(h/ctu).                    */
int vvcb_ctu_hads_islice(vvcb_ctx* ctx, int32_t* out, int n_ctus);

/* vvcb_features_eval: the 27 classifier inputs of the fork's FAST_ALGORITHM block (EL/EncCu.cpp:72-164, 816-1138).
 * The host walk owns the coding structure, so it ships the current CU and the neighbour CUs it found with
 * tempCS->getCU (:857-933: left, left-down, up, right-up, left-up; only their area and depths are used); the engine
 * computes every pixel-derived term from the frame's (LMCS-mapped) original luma, saturated to 8 bit as the
 * reference's convertTo(CV_8U) does.                                                                                 */
#define VVCB_NUM_FEATURES 27
typedef struct vvcb_feat_cu {
  int16_t x, y;             /* luma position                                                                        */
  uint8_t w, h;             /* luma size, powers of two 4..128                                                      */
  uint8_t qt_depth, mt_depth;
} vvcb_feat_cu;
typedef struct vvcb_feat_job {
  vvcb_feat_cu cu;          /* currCsArea + partitioner.currQtDepth / currMtDepth                                   */
  uint8_t n_neighbours;     /* valid_num (0..5); the reference evaluates the classifier only when it is >= 3        */
  uint8_t pad[7];
  vvcb_feat_cu nb[5];
} vvcb_feat_job;
typedef struct vvcb_feat_result {
  int32_t f[VVCB_NUM_FEATURES];   /* features[0..26] (EL/EncCu.cpp:1098-1138); neighbour terms are 0 when n_neighbours == 0 */
  int32_t valid;                  /* n_neighbours >= 3                                                              */
} vvcb_feat_result;
int vvcb_features_eval(vvcb_ctx* ctx, const vvcb_feat_job* jobs, int n, vvcb_feat_result* results);

/* ---- raw device memory for resident benchmarking --------------------------------------------- */
int vvcb_dev_alloc(vvcb_ctx* ctx, size_t bytes, void** out);
int vvcb_dev_free (vvcb_ctx* ctx, void* p);
int vvcb_host_alloc(vvcb_ctx* ctx, size_t bytes, void** out);   /* page-locked host memory */
int vvcb_host_free (vvcb_ctx* ctx, void* p);
int vvcb_dev_upload  (vvcb_ctx* ctx, void* dst, const void* src, size_t bytes);
int vvcb_dev_download(vvcb_ctx* ctx, void* dst, const void* src, size_t bytes);
int vvcb_sync(vvcb_ctx* ctx);
/* CUDA-event timing on the context's own stream (torch.cuda.Event cannot see it).               */
int vvcb_timer_start(vvcb_ctx* ctx);
int vvcb_timer_stop (vvcb_ctx* ctx, float* ms);
/* Per-kernel device time (CUDA events on the context's stream around each launch), accumulated since
 * the last call; enable with on != 0.  ms[0] plan, ms[1] eval (prediction+SAD+SATD), ms[2] lists.   */
int vvcb_kernel_timing(vvcb_ctx* ctx, int on);
int vvcb_kernel_times(vvcb_ctx* ctx, float ms[3], int* launches);
/* same for vvcb_tu_eval / vvcb_tu_eval_pred: ms[0] (prediction +) transform pass, ms[1] quantiser kernels, ms[2] reconstruction pass,
 * ms[3] residual rate estimation                                                                                         */
int vvcb_tu_kernel_times(vvcb_ctx* ctx, float ms[4], int* calls);
/* Integer-ALU roofline denominator, measured live: dependent-free IMAD / IADD3+LOP3 / 1:1 mixed
 * instruction streams on every SM; results in 10^9 lane-operations per second.                  */
int vvcb_measure_int_peak(vvcb_ctx* ctx, double* gops_imad, double* gops_alu, double* gops_mixed);
/* kernel launches issued by this context since creation (bench.py reports the delta).           */
uint64_t vvcb_launch_count(const vvcb_ctx* ctx);
/* Where the host time of vvcb_cu_eval goes, cumulative wall-clock nanoseconds since the context was created: ns[0] packing the
 * rectangles and launching the rough mode decision, ns[1] waiting for its lists (calls with candidate templates only), ns[2] expanding
 * the templates and assembling the TU batch, ns[3] launching the TU stage, ns[4] waiting for its results, ns[5] handing the outputs
 * back; then two spans on the device (CUDA events on the context's stream): ns[6] rough mode decision, ns[7] TU stage.  A measuring
 * aid for the latency-bound use (profiles/).                                                                                     */
int vvcb_cu_eval_phases(const vvcb_ctx* ctx, uint64_t ns[8], uint64_t* calls);

#ifdef __cplusplus
}
#endif
#endif
