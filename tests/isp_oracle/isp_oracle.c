/*
 * TEST INFRASTRUCTURE -- plain-C restatement of the luma evaluation of one intra sub-partition (ISP) candidate whose transform blocks are
 * all at least 4x4: IntraSearch::xIntraCodingLumaISP (EL/IntraSearch.cpp:3171) on one restored estimator.  Built on the oracle's pinned
 * components (oracle/vvc_oracle*.c): reference-line padding (orc_ref_fill), prediction (orc_pred_regular and the angular restatement
 * below, which differs from the oracle's only in the ISP reference-line lengths), transforms, quantisers, reconstruction and the
 * residual rate.
 *
 * Parity status: the components are pinned; the chaining (line hand-over, cbf and context carry) is restated from the cited reference
 * lines and NOT compared with the reference encoder's own ISP output.
 */
#include <stdlib.h>
#include <string.h>
#include "vvc_oracle.h"
#include "../vvc_intra_b200/csrc/vvc_rom_tables.h"

uint64_t orc_residual_bits_carry(const int32_t* coeff, int w, int h, int mts_idx, int ts_allowed, int mts_allowed, int dep_quant,
                                 const vvcb_ctx_states* states, vvcb_ctx_states* carry);
void orc_tr_types_mts(int mts_idx, int* hor, int* ver);

static int imin(int a, int b) { return a < b ? a : b; }
static int imax(int a, int b) { return a > b ? a : b; }
static int ilog2(int v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }
static int iclip(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

/* transform pair of the block being coded (hor | ver << 2), -1: from mts_idx (TrQuant::getTrTypes, CL/TrQuant.cpp:752-783) */
static int g_pair = -1;
void orc_tr_types(int mts_idx, int* hor, int* ver)
{
  if (g_pair >= 0) { *hor = g_pair & 3; *ver = g_pair >> 2; return; }
  orc_tr_types_mts(mts_idx, hor, ver);
}

/* PartitionerImpl::getTUIntraSubPartitions (CL/UnitPartitioner.cpp:978): equal blocks of at least 16 samples along the split */
int orc_isp_blocks(int cu_w, int cu_h, int hor, int* bw, int* bh)
{
  const int split = hor ? cu_h : cu_w, other = hor ? cu_w : cu_h;
  const int floorSize = other < 16 ? 16 / other : 1;
  const int size = imax(split >> 2, floorSize);
  *bw = hor ? cu_w : size; *bh = hor ? size : cu_h;
  return split / size;
}

/* IntraPrediction::initIntraPatternChTypeISP (CL/IntraPrediction.cpp:1136-1203), written as the reference does it: block 0 takes the
 * lines of one xFillReferenceSamples over the CU (top 2*cu_w, left 2*cu_h samples); block k > 0 of a horizontal split shifts that left
 * column down by k block heights and takes as its top line block k-1's last row, repeated past the CU; a vertical split does the same
 * with the top row and block k-1's last column.  Without the left (horizontal) / above (vertical) neighbour the shifted side and the
 * corner take the first sample of the new line.  cu_reco: the candidate's blocks 0..k-1 in coding order, each dense bw*bh.
 * top: m_topRefLength + 1 = cu_w + bw + 1 samples, left: cu_h + bh + 1; top[0] == left[0]. */
void orc_isp_lines(const int16_t* pic, int stride, int bd, int x, int y, int cu_w, int cu_h, int hor, int k,
                   int avail_al, int n_above, int n_above_right, int n_left, int n_below_left,
                   const int16_t* cu_reco, int16_t* top, int16_t* left)
{
  int16_t ftop[2 * 64 + 1], fleft[2 * 64 + 1];
  int bw, bh, i;
  orc_isp_blocks(cu_w, cu_h, hor, &bw, &bh);
  {
    const int T = cu_w + bw, L = cu_h + bh, bs = bw * bh;
    orc_ref_fill(pic, stride, x, y, cu_w, cu_h, 0, bd, avail_al, n_above, n_above_right, n_left, n_below_left, ftop, fleft);
    if (k == 0) {
      for (i = 0; i <= T; i++) top[i] = ftop[i];
      for (i = 0; i <= L; i++) left[i] = fleft[i];
      return;
    }
    if (hor) {
      const int16_t* last = cu_reco + (size_t)(k - 1) * bs + (bh - 1) * bw;     /* block k-1's last row */
      for (i = 0; i <= L; i++) left[i] = fleft[i + k * bh];
      for (i = 1; i <= T; i++) top[i] = last[imin(i - 1, cu_w - 1)];
      if (!n_left) for (i = 0; i <= L; i++) left[i] = top[1];
      top[0] = left[0];
    } else {
      const int16_t* prev = cu_reco + (size_t)(k - 1) * bs;                     /* block k-1: its last column */
      for (i = 0; i <= T; i++) top[i] = ftop[i + k * bw];
      for (i = 1; i <= L; i++) left[i] = prev[imin(i - 1, cu_h - 1) * bw + bw - 1];
      if (!n_above) for (i = 0; i <= T; i++) top[i] = left[1];
      left[0] = top[0];
    }
  }
}

/* initPredIntraParams for an ISP block (CL/IntraPrediction.cpp:492-511, :544-551, :558-574): the CU's wide-angle remap, the block's
 * PDPC, unfiltered lines, cubic interpolation */
void orc_isp_ipa(int cu_w, int cu_h, int bw, int bh, int mode, orc_ipa* p)
{
  orc_ipa_init(cu_w, cu_h, mode, 1, 0, p);     /* reference line 1: angles only, no filters, no PDPC */
  p->mrl = 0; p->ref_filter = 0; p->interp = 0;
  p->pdpc = bw >= 4 && bh >= 4;
  p->ang_scale = 0;
  if (mode > 1 && p->angle < 0) p->pdpc = 0;
  else if (mode > 1 && p->angle > 0) {
    p->ang_scale = imin(2, ilog2(p->is_ver ? bh : bw) - (ilog2(3 * p->inv_angle - 2) - 8));
    p->pdpc = p->pdpc && p->ang_scale >= 0;
  }
}

/* xPredIntraAng (CL/IntraPrediction.cpp:633-935) with the ISP line lengths: the main reference of a positive angle holds
 * m_topRefLength / m_leftRefLength samples and is extended by replicating the last one (:717-726). */
static void pred_angular_isp(const int16_t* top, const int16_t* left, int T, int L, int w, int h, int bd, const orc_ipa* p, int16_t* pred)
{
  const int16_t* mainSrc = p->is_ver ? top : left;
  const int16_t* sideSrc = p->is_ver ? left : top;
  const int mw = p->is_ver ? w : h, mh = p->is_ver ? h : w;
  const int mainLen = p->is_ver ? T : L, sideLen = p->is_ver ? L : T;
  const int angle = p->angle, maxv = (1 << bd) - 1;
  int16_t mainBuf[512], sideBuf[512];
  int16_t* refMain = mainBuf + 128;
  int16_t* refSide = sideBuf;
  int i, r, c;
  if (angle < 0) {
    for (i = 0; i <= mw + 1; i++) refMain[i] = mainSrc[i];
    for (i = 0; i <= mh + 1; i++) refSide[i] = sideSrc[i];
    for (i = -mh; i <= -1; i++) refMain[i] = refSide[imin((-i * p->inv_angle + 256) >> 9, mh)];
  } else {
    for (i = 0; i <= mainLen; i++) refMain[i] = mainSrc[i];
    for (i = 0; i <= sideLen; i++) refSide[i] = sideSrc[i];
    for (i = 1; i <= 2; i++) refMain[mainLen + i] = refMain[mainLen];
  }
  for (r = 0; r < mh; r++) {
    int line[64];
    if (angle == 0) {
      for (c = 0; c < mw; c++) line[c] = refMain[c + 1];
      if (p->pdpc) {
        const int scale = (ilog2(mw) + ilog2(mh) - 2) >> 2;
        const int lim = imin(3 << scale, mw);
        for (c = 0; c < lim; c++) {
          const int wL = 32 >> ((2 * c) >> scale);
          line[c] = iclip(line[c] + ((wL * (refSide[1 + r] - refMain[0]) + 32) >> 6), 0, maxv);
        }
      }
    } else {
      const int pos = angle * (r + 1);
      const int dInt = pos >> 5, dFrac = pos & 31;
      if (abs(angle) & 31) {
        const int8_t* f = kIntraCubicFilter + 4 * dFrac;
        for (c = 0; c < mw; c++) {
          const int16_t* q = refMain + dInt + c;
          line[c] = iclip((f[0] * q[0] + f[1] * q[1] + f[2] * q[2] + f[3] * q[3] + 32) >> 6, 0, maxv);
        }
      } else {
        for (c = 0; c < mw; c++) line[c] = refMain[c + dInt + 1];
      }
      if (p->pdpc) {
        const int scale = p->ang_scale;
        const int lim = imin(3 << scale, mw);
        int acc = 256;
        for (c = 0; c < lim; c++) {
          int wL, l;
          acc += p->inv_angle;
          wL = 32 >> ((2 * c) >> scale);
          l = refSide[r + (acc >> 9) + 1];
          line[c] = line[c] + ((wL * (l - line[c]) + 32) >> 6);
        }
      }
    }
    for (c = 0; c < mw; c++) {
      if (p->is_ver) pred[r * w + c] = (int16_t)line[c];
      else           pred[c * w + r] = (int16_t)line[c];
    }
  }
}

void orc_isp_pred(const int16_t* top, const int16_t* left, int cu_w, int cu_h, int bw, int bh, int bd, int mode, int16_t* pred)
{
  orc_ipa p;
  orc_isp_ipa(cu_w, cu_h, bw, bh, mode, &p);
  if (mode < 2) orc_pred_regular(top, left, bw, bh, bd, mode, &p, pred);
  else pred_angular_isp(top, left, cu_w + bw, cu_h + bh, bw, bh, bd, &p, pred);
}

/* TBitEstimator::encodeBin on one model: price, then BinProbModel_Std::update (CL/Contexts.h:104-131) */
static uint32_t code_bin(vvcb_bin_model* m, unsigned bin)
{
  const int rate0 = m->rate >> 4, rate1 = m->rate & 15;
  const uint32_t bits = kBinFracBits[2 * ((unsigned)(m->state[0] + m->state[1]) >> 8) + bin];
  m->state[0] = (uint16_t)(m->state[0] - ((m->state[0] >> rate0) & 0x7fe0));
  m->state[1] = (uint16_t)(m->state[1] - ((m->state[1] >> rate1) & 0x7ffe));
  if (bin) {
    m->state[0] = (uint16_t)(m->state[0] + ((0x7fffu >> rate0) & 0x7fe0));
    m->state[1] = (uint16_t)(m->state[1] + ((0x7fffu >> rate1) & 0x7ffe));
  }
  return bits;
}

/* BinFracBits::intBits of every context the dependent quantiser reads (vvcb_dq_rates lists the models of vvcb_ctx_states behind mts_idx) */
void orc_rates_from_states(const vvcb_ctx_states* s, vvcb_dq_rates* r)
{
  const vvcb_bin_model* m = (const vvcb_bin_model*)s + 11;
  uint32_t* o = (uint32_t*)r;
  const int n = (int)(sizeof(vvcb_dq_rates) / (2 * sizeof(uint32_t)));
  int i;
  for (i = 0; i < n; i++) {
    const unsigned q = (unsigned)(m[i].state[0] + m[i].state[1]) >> 8;
    o[2 * i] = kBinFracBits[2 * q]; o[2 * i + 1] = kBinFracBits[2 * q + 1];
  }
}

/* One candidate.  org / pic: original and reconstruction planes (stride); dep_quant: slice->getDepQuantEnabledFlag().  pred / level / reco:
 * cu_w*cu_h each, blocks in coding order.  Per block k: carried[k] = the residual models after it, cbf_delta[k] = its cbfDeltaBits.
 * Returns the number of blocks. */
int orc_isp_chain(const int16_t* org, const int16_t* pic, int stride, int bd, int dep_quant, const vvcb_rmd_visit* v, const vvcb_isp_job* j,
                  const vvcb_ctx_states* states, int16_t* pred, int32_t* level, int16_t* reco, vvcb_isp_result* res,
                  vvcb_ctx_states* carried, int32_t* cbf_delta)
{
  const int cu_w = 1 << v->log2w, cu_h = 1 << v->log2h, hor = j->isp_mode == VVCB_ISP_HOR;
  const int dq = (j->flags & VVCB_TU_DEPQUANT) != 0, rate = (j->flags & VVCB_TU_RATE) != 0;
  const int qp = j->qp_per * 6 + j->qp_rem;
  int bw, bh, k, i, any = 0;
  const int np = orc_isp_blocks(cu_w, cu_h, hor, &bw, &bh);
  const int bs = bw * bh;
  vvcb_bin_model cbfCtx[2];
  vvcb_ctx_states cur;
  int16_t top[2 * 64 + 3], left[2 * 64 + 3], resi[64 * 64], resi2[64 * 64];
  int32_t coeff[64 * 64], deq[64 * 64];
  uint8_t cbf[4] = { 0, 0, 0, 0 };
  memset(res, 0, sizeof(*res));
  cbfCtx[0] = j->cbf[0]; cbfCtx[1] = j->cbf[1];
  if (states) cur = *states; else memset(&cur, 0, sizeof(cur));
  res->n_parts = (uint8_t)np;
  for (k = 0; k < np; k++) {
    const int bx = hor ? 0 : k * bw, by = hor ? k * bh : 0;
    const int pair = (j->use_mts && bw <= 16 ? VVCB_TR_DST7 : VVCB_TR_DCT2) | (j->use_mts && bh <= 16 ? VVCB_TR_DST7 : VVCB_TR_DCT2) << 2;
    const int16_t* o = org + (size_t)(v->y + by) * stride + v->x + bx;
    int16_t* pk = pred + k * bs;
    int32_t* lk = level + k * bs;
    const int last = k == np - 1, inferred = last && !any;
    const int ctxId = k ? cbf[k - 1] : 0;                                   /* Ctx::QtCbf[luma](2 + cbf of the previous block) */
    int32_t delta = 0;
    int absSum, sumCoeff = 0;
    orc_isp_lines(pic, stride, bd, v->x, v->y, cu_w, cu_h, hor, k, v->avail_al, v->n_above, v->n_above_right, v->n_left, v->n_below_left,
                  reco, top, left);
    orc_isp_pred(top, left, cu_w, cu_h, bw, bh, bd, j->mode, pk);
    for (i = 0; i < bs; i++) resi[i] = (int16_t)(o[(i / bw) * stride + i % bw] - pk[i]);
    g_pair = pair;
    orc_fwd_transform(resi, bw, bw, bh, bd, 0, coeff);
    for (i = 0; i < bs; i++) sumCoeff += abs(coeff[i]);
    if (!inferred) {                                                        /* RateEstimator::xSetLastCoeffOffset, ISP branch */
      const unsigned q = (unsigned)(cbfCtx[ctxId].state[0] + cbfCtx[ctxId].state[1]) >> 8;
      delta = (int32_t)kBinFracBits[2 * q + 1] - (int32_t)kBinFracBits[2 * q];
    }
    if (cbf_delta) cbf_delta[k] = delta;
    if (dq) {
      vvcb_dq_rates r;
      orc_rates_from_states(&cur, &r);
      absSum = orc_dep_quant(coeff, bw, bh, bd, 0, 0, qp, j->lambda, &r, delta, lk);
      orc_dep_dequant(lk, bw, bh, bd, qp, deq);
    } else {
      absSum = orc_quant_scalar(coeff, bw, bh, bd, j->qp_per, j->qp_rem, 0, lk);
      orc_dequant(lk, bw, bh, bd, j->qp_per, j->qp_rem, 0, deq);
    }
    orc_inv_transform(deq, bw, bh, bd, 0, resi2, bw);
    g_pair = -1;
    res->part[k].abs_sum_coeff = sumCoeff;
    res->part[k].abs_sum_level = absSum;
    res->part[k].sse = orc_reconstruct_sse(o, stride, pk, resi2, bw, bh, bd, reco + k * bs);
    {
      int nz = 0;
      for (i = 0; i < bs; i++) nz |= lk[i] != 0;
      cbf[k] = (uint8_t)nz;
    }
    /* xGetIntraFracBitsQT: the cbf bin (not coded when inferred), then residual_coding of a coded block on the same estimator */
    res->cbf_bits[k] = inferred ? 0u : code_bin(&cbfCtx[ctxId], cbf[k]);
    res->cbf[k] = cbf[k];
    any |= cbf[k];
    if (dq || rate) {
      const uint64_t bits = orc_residual_bits_carry(lk, bw, bh, 0, 0, 0, dep_quant, &cur, &cur);
      if (rate) res->part[k].frac_bits = bits;
    }
    if (carried) carried[k] = cur;
  }
  res->discarded = (uint8_t)!any;
  return np;
}
