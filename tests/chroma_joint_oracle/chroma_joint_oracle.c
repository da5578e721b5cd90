/*
 * TEST INFRASTRUCTURE -- plain-C chain of one joint Cb-Cr candidate (the checker of vvcb_chroma_joint_tu_eval), composed from the functions
 * the chain of vvcb_chroma_tu_eval uses (tests/chroma_tu_oracle/chroma_tu_oracle.c, whose library this one links): the chroma prediction of
 * oracle/vvc_oracle_chroma.c, the oracle's DCT-II, scalar or chroma dependent quantisation, dequantisation and inverse transform of the
 * combined residual, the inverse mapping, both reconstructions and SSEs, and the cbf, joint-flag and chroma residual bins on one carried
 * copy of the models.  Parity status: UNPINNED.
 */
#include <stdlib.h>
#include <string.h>
#include "../../oracle/vvc_oracle_chroma.h"
#include "../../vvc_intra_b200/csrc/vvc_rom_tables.h"

/* from libchroma_tu_oracle.so */
int orc_dep_quant_chroma(const int32_t* coeff, int w, int h, int bd, int mts_idx, int lfnst_idx, int qp, double lambda,
                         const vvcb_dq_rates* rates, int cbf_delta_bits, int32_t* level);
void orc_chroma_dq_rates(const vvcb_chroma_ctx_states* st, vvcb_dq_rates* r);
int32_t orc_chroma_cbf_delta_bits(const vvcb_bin_model* m);
uint64_t orc_chroma_residual_bits(const int32_t* level, int w, int h, int dep_quant, vvcb_chroma_ctx_states* c);

/* TBitEstimator::encodeBin: price, then BinProbModel_Std::update */
static uint32_t code_bin(vvcb_bin_model* m, unsigned bin)
{
  const uint32_t b = kBinFracBits[2 * (((unsigned)m->state[0] + m->state[1]) >> 8) + bin];
  const int rate0 = m->rate >> 4, rate1 = m->rate & 15;
  m->state[0] = (uint16_t)(m->state[0] - ((m->state[0] >> rate0) & 0x7fe0));
  m->state[1] = (uint16_t)(m->state[1] - ((m->state[1] >> rate1) & 0x7ffe));
  if (bin) {
    m->state[0] = (uint16_t)(m->state[0] + ((0x7fffu >> rate0) & 0x7fe0));
    m->state[1] = (uint16_t)(m->state[1] + ((0x7fffu >> rate1) & 0x7ffe));
  }
  return b;
}

/* The forward combination is the library's restatement of the encoder derivation of JVET-O0105 (H.266 does not specify it; C division,
 * truncating toward zero); the inverse mapping is H.266 8.7.2 under TuCResMode, in int. */
int orc_chroma_joint_combine(int cb, int cr, int mode, int sign)
{
  switch (mode) {
  case 1: return (4 * cb + 2 * sign * cr) / 5;
  case 2: return (cb + sign * cr) / 2;
  default: return (4 * cr + 2 * sign * cb) / 5;
  }
}

void orc_chroma_joint_inverse(const int16_t* r, int n, int mode, int sign, int32_t* cb, int32_t* cr)
{
  int i;
  for (i = 0; i < n; i++) {
    const int v = r[i];
    switch (mode) {
    case 1: cb[i] = v; cr[i] = (sign * v) >> 1; break;
    case 2: cb[i] = v; cr[i] = sign * v; break;
    default: cb[i] = (sign * v) >> 1; cr[i] = v; break;
    }
  }
}

/* One joint candidate, as orc_chroma_tu_cand: the prediction of both components, the combined residual coded as Cb is there (cbfDeltaBits
 * from Ctx::QtCbf[Cr](0) for mode 3, else Ctx::QtCbf[Cb](0)), the inverse mapping, both reconstructions and SSEs; with VVCB_TU_RATE and a
 * level, tu_cb_coded_flag, tu_cr_coded_flag, tu_joint_cbcr_residual_flag and residual_coding on one carried copy of the models.
 * level / reco / pred: 2 w*h each (level: the coded residual's, then zeros; reco / pred: Cb, then Cr). */
void orc_chroma_joint_tu_cand(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu, int dep_quant,
                              const vvcb_chroma_visit* v, const vvcb_chroma_joint_tu_job* j, const vvcb_chroma_joint_ctx_states* states,
                              int32_t* level, int16_t* reco, int16_t* pred, vvcb_chroma_joint_tu_result* out)
{
  const int w = 1 << v->log2w, h = 1 << v->log2h, n = w * h;
  const int dq = (j->flags & VVCB_TU_DEPQUANT) != 0, rate = (j->flags & VVCB_TU_RATE) != 0;
  const int qp = 6 * j->qp_per + j->qp_rem;
  int16_t* all = (int16_t*)malloc(sizeof(int16_t) * 16 * n);
  int16_t* resi = (int16_t*)malloc(sizeof(int16_t) * n);
  int32_t* coeff = (int32_t*)malloc(sizeof(int32_t) * n);
  int32_t* deq = (int32_t*)malloc(sizeof(int32_t) * n);
  int32_t* res = (int32_t*)malloc(sizeof(int32_t) * 2 * n);
  vvcb_chroma_result pr;
  vvcb_chroma_joint_ctx_states start, carry;
  vvcb_dq_rates rates;
  int c, x, y, absSum;
  memset(out, 0, sizeof(*out));
  if (states) start = *states; else memset(&start, 0, sizeof(start));
  carry = start;
  orc_chroma_visit(planes, cstride, luma, lstride, bd, ctu, v, &pr, all);
  memcpy(pred, all + (size_t)j->cand * 2 * n, sizeof(int16_t) * 2 * n);
  for (y = 0; y < h; y++)
    for (x = 0; x < w; x++) {
      const int s = y * w + x;
      const int rcb = planes[0][(size_t)(v->y + y) * cstride + v->x + x] - pred[s];
      const int rcr = planes[1][(size_t)(v->y + y) * cstride + v->x + x] - pred[n + s];
      resi[s] = (int16_t)orc_chroma_joint_combine(rcb, rcr, j->mode, j->sign);
    }
  orc_fwd_transform(resi, w, w, h, bd, 0, coeff);
  out->res.abs_sum_coeff = orc_abs_sum_for_preselection(coeff, w, h, 0);
  if (dq) {
    const int32_t delta = orc_chroma_cbf_delta_bits(j->mode == 3 ? &start.chroma.cbf_cr[0] : &start.chroma.cbf_cb[0]);
    orc_chroma_dq_rates(&start.chroma, &rates);
    absSum = orc_dep_quant_chroma(coeff, w, h, bd, 0, 0, qp, j->lambda, &rates, delta, level);
    orc_dep_dequant(level, w, h, bd, qp, deq);
  } else {
    absSum = orc_quant_scalar(coeff, w, h, bd, j->qp_per, j->qp_rem, 0, level);
    orc_dequant(level, w, h, bd, j->qp_per, j->qp_rem, 0, deq);
  }
  memset(level + n, 0, sizeof(int32_t) * n);
  out->res.abs_sum_level = absSum;
  out->cbf = absSum != 0;
  orc_inv_transform(deq, w, h, bd, 0, resi, w);
  orc_chroma_joint_inverse(resi, n, j->mode, j->sign, res, res + n);
  for (c = 0; c < 2; c++) {
    uint64_t sse = 0;
    for (y = 0; y < h; y++)
      for (x = 0; x < w; x++) {
        const int s = y * w + x, maxv = (1 << bd) - 1;
        int rec = pred[c * n + s] + res[c * n + s];
        rec = rec < 0 ? 0 : rec > maxv ? maxv : rec;
        const int d = planes[c][(size_t)(v->y + y) * cstride + v->x + x] - rec;
        reco[c * n + s] = (int16_t)rec;
        sse += (uint64_t)((int64_t)d * d);
      }
    out->sse[c] = sse;
  }
  if (rate && out->cbf) {                              /* transform_unit order: cbf Cb, cbf Cr, joint flag, residual */
    const unsigned cbfCb = j->mode != 3, cbfCr = j->mode != 1;
    out->cbf_bits[0] = code_bin(&carry.chroma.cbf_cb[0], cbfCb);
    out->cbf_bits[1] = code_bin(&carry.chroma.cbf_cr[cbfCb], cbfCr);
    out->joint_bits = code_bin(&carry.joint[2 * cbfCb + cbfCr - 1], 1);
    out->res.frac_bits = orc_chroma_residual_bits(level, w, h, dep_quant, &carry.chroma);
  }
  free(all); free(resi); free(coeff); free(deq); free(res);
}

void orc_chroma_joint_tu_batch(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu, int dep_quant,
                               const vvcb_chroma_visit* visits, const vvcb_chroma_joint_tu_job* jobs, int n,
                               const vvcb_chroma_joint_ctx_states* states, int32_t* level, int16_t* reco, int16_t* pred,
                               vvcb_chroma_joint_tu_result* out)
{
  int i;
  for (i = 0; i < n; i++) {
    const vvcb_chroma_joint_tu_job* j = &jobs[i];
    const int carried = (j->flags & (VVCB_TU_DEPQUANT | VVCB_TU_RATE)) != 0;
    orc_chroma_joint_tu_cand(planes, cstride, luma, lstride, bd, ctu, dep_quant, &visits[j->visit], j, carried ? &states[j->rate_idx] : NULL,
                             level + j->offset, reco + j->offset, pred + j->offset, &out[i]);
  }
}
