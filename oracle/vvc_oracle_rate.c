/*
 * TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the reference's residual rate estimation for a luma TU
 * (SURVEY.md 8f-2): CABACWriter::residual_coding on the bit estimator (EL/CABACWriter.cpp:3773-3895) with mts_coding
 * (:3897-3950), last_sig_coeff (:3960-4020), residual_coding_subblock (:4164-4300), residual_codingTS /
 * residual_coding_subblockTS (:4025-4160, :4305-4520), the context derivations of CoeffCodingContext
 * (CL/ContextModelling.h, CL/ContextModelling.cpp:40-134), the adaptive bin model BinProbModel_Std (CL/Contexts.h:90-163) and
 * the estimator's bypass / Golomb-Rice pricing (EL/BinEncoder.cpp encodeRemAbsEP).  No sign hiding (off with dependent
 * quantisation), no BDPCM, no ISP.  See vvc_oracle.h for who may use it.
 *
 * Parity status: PINNED ('C' records of oracle/ref_trace_hooks.cpp: context states in, fractional bits out;
 * tests/test_oracle_rate.py).
 */
#include <stdlib.h>
#include <string.h>
#include "vvc_oracle.h"
#include "../vvc_intra_b200/csrc/vvc_rom_tables.h"

#define EP_BITS (1u << 15)

static int imin(int a, int b) { return a < b ? a : b; }
static int imax(int a, int b) { return a > b ? a : b; }
static int ilog2(int v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }

static const uint8_t kGroupIdx[32] = { 0,1,2,3,4,4,5,5,6,6,6,6,7,7,7,7,8,8,8,8,8,8,8,8,9,9,9,9,9,9,9,9 };
static const uint8_t kMinInGroup[14] = { 0,1,2,3,4,6,8,12,16,24,32,48,64,96 };
static const uint8_t kRicePars[32] = { 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 3, 3, 3 };
static const uint8_t kRicePos0[3][32] = {
  {0, 0, 0, 0, 0, 1, 2,    2, 2, 2, 2, 2, 4, 4,    4, 4, 4, 4,  4,  4,  4,  4,  4,  8,  8,  8,  8,  8,     8,  8,  8,  8},
  {1, 1, 1, 1, 2, 3, 4,    4, 4, 6, 6, 6, 8, 8,    8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 12, 16, 16,    16, 16, 16, 16},
  {1, 1, 2, 2, 2, 3, 4,    4, 4, 6, 6, 6, 8, 8,    8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 16, 16, 16,    16, 16, 16, 16} };
static const uint8_t kTsRicePars[32] = { 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2 };

typedef struct { uint64_t bits; } est;

/* TBitEstimator::encodeBin -> BinProbModel_Std::estFracBitsUpdate (CL/Contexts.h:104-131); MASK_0 = 0x7fe0, MASK_1 = 0x7ffe */
static void code_bin(est* e, vvcb_bin_model* m, unsigned bin)
{
  const int rate0 = m->rate >> 4, rate1 = m->rate & 15;
  const unsigned state = (unsigned)(m->state[0] + m->state[1]) >> 8;
  e->bits += kBinFracBits[2 * state + bin];
  m->state[0] = (uint16_t)(m->state[0] - ((m->state[0] >> rate0) & 0x7fe0));
  m->state[1] = (uint16_t)(m->state[1] - ((m->state[1] >> rate1) & 0x7ffe));
  if (bin) {
    m->state[0] = (uint16_t)(m->state[0] + ((0x7fffu >> rate0) & 0x7fe0));
    m->state[1] = (uint16_t)(m->state[1] + ((0x7fffu >> rate1) & 0x7ffe));
  }
}

/* BitEstimatorBase::encodeRemAbsEP (EL/BinEncoder.cpp), maxLog2TrDynamicRange 15 */
static void code_rem_abs_ep(est* e, unsigned bins, unsigned rice)
{
  const unsigned threshold = 5u << rice;
  if (bins < threshold) e->bits += (uint64_t)((bins >> rice) + 1 + rice) * EP_BITS;
  else {
    const unsigned maxPrefix = 32 - 5 - 15;
    unsigned prefix = 0, code = (bins >> rice) - 5, suffix;
    if (code >= ((1u << maxPrefix) - 1)) { prefix = maxPrefix; suffix = 15; }
    else { while (code > ((2u << prefix) - 2)) prefix++; suffix = prefix + rice + 1; }
    e->bits += (uint64_t)(5 + prefix + suffix) * EP_BITS;
  }
}

typedef struct {
  int w, h, numCoeff, gw, gh;
  uint16_t idx[1024]; uint8_t x[1024], y[1024];
  uint16_t sbbPos[64];
} res_scan;

static void build_res_scan(res_scan* s, int w, int h)
{
  int gx[64], gy[64], ix[16], iy[16], n, d, y, g, i;
  const int nzW = imin(32, w), nzH = imin(32, h);
  s->w = w; s->h = h; s->gw = nzW >> 2; s->gh = nzH >> 2; s->numCoeff = nzW * nzH;
  for (n = 0, d = 0; d <= s->gw + s->gh - 2; d++) for (y = imin(d, s->gh - 1); y >= imax(0, d - s->gw + 1); y--) { gx[n] = d - y; gy[n] = y; n++; }
  for (n = 0, d = 0; d <= 6; d++) for (y = imin(d, 3); y >= imax(0, d - 3); y--) { ix[n] = d - y; iy[n] = y; n++; }
  for (g = 0; g < s->gw * s->gh; g++) {
    s->sbbPos[g] = (uint16_t)(gy[g] * s->gw + gx[g]);
    for (i = 0; i < 16; i++) {
      const int px = gx[g] * 4 + ix[i], py = gy[g] * 4 + iy[i];
      s->x[g * 16 + i] = (uint8_t)px; s->y[g * 16 + i] = (uint8_t)py; s->idx[g * 16 + i] = (uint16_t)(py * w + px);
    }
  }
}

/* CABACWriter::mts_coding (:3897-3950), JVET_O0294 on */
static void mts_coding(est* e, vvcb_ctx_states* c, int mts_idx, int ts_allowed, int mts_allowed)
{
  if (!mts_allowed && !ts_allowed) return;
  if (ts_allowed) code_bin(e, &c->mts_idx[6], mts_idx == 1);
  if (mts_idx != 1 && mts_allowed) {
    const unsigned symbol = mts_idx != 0;
    code_bin(e, &c->mts_idx[0], symbol);
    if (symbol) {
      int i, ctx = 7;
      for (i = 0; i < 3; i++, ctx++) {
        const unsigned s2 = mts_idx > i + 2;
        code_bin(e, &c->mts_idx[ctx], s2);
        if (!s2) break;
      }
    }
  }
}

/* template sums of CoeffCodingContext::sigCtxIdAbs / templateAbsSum (CL/ContextModelling.h:102-196) */
static void template_sums(const int32_t* coeff, int w, int h, int px, int py, int* sumAbs1, int* numPos, int* sumAbs)
{
  const int32_t* p = coeff + py * w + px;
  int s1 = 0, np = 0, sa = 0, a;
#define UPD(v) { a = abs(v); s1 += imin(4 + (a & 1), a); np += !!a; sa += a; }
  if (px < w - 1) {
    UPD(p[1]);
    if (px < w - 2) UPD(p[2]);
    if (py < h - 1) UPD(p[w + 1]);
  }
  if (py < h - 1) {
    UPD(p[w]);
    if (py < h - 2) UPD(p[2 * w]);
  }
#undef UPD
  *sumAbs1 = s1; *numPos = np; *sumAbs = sa;
}

static void residual_ts(est* e, vvcb_ctx_states* c, const res_scan* sc, const int32_t* coeff)
{
  const int w = sc->w, numSbb = sc->gw * sc->gh;
  uint8_t sigGroup[64], coded[64];
  int remCtxBins = 2 * sc->w * sc->h, sb, i;
  memset(coded, 0, sizeof(coded));
  for (sb = 0; sb < numSbb; sb++) {
    sigGroup[sb] = 0;
    for (i = 0; i < 16; i++) if (coeff[sc->idx[sb * 16 + i]]) sigGroup[sb] = 1;
  }
  for (sb = 0; sb < numSbb; sb++) {
    const int sbPos = sc->sbbPos[sb], sy = sbPos / sc->gw, sx = sbPos - sy * sc->gw;
    int anyEarlier = 0, k, numNonZero = 0;
    /* initSubblock: m_sigCoeffGroupFlag holds the flags of the sub-blocks initialised so far, by raster position */
    coded[sbPos] = sigGroup[sb];
    {
      const int sigLeft = sx > 0 ? coded[sbPos - 1] : 0, sigAbove = sy > 0 ? coded[sbPos - sc->gw] : 0;
      vvcb_bin_model* mSbb = &c->ts_sig_sbb[sigLeft + sigAbove];
      /* only1stSigGroup(): no flag set except possibly the one of the last sub-block in scan order */
      for (k = 0; k < numSbb; k++) if (coded[k] && k != sc->sbbPos[numSbb - 1]) anyEarlier = 1;
      if (sb != numSbb - 1 || anyEarlier) {
        code_bin(e, mSbb, sigGroup[sb]);
        if (!sigGroup[sb]) continue;
      }
    }
    for (i = 0; i < 16; i++) {                                   /* first pass: sig, sign, gt1, parity */
      const int pos = sb * 16 + i, px = sc->x[pos], py = sc->y[pos];
      const int32_t v = coeff[sc->idx[pos]];
      const int left = px > 0 ? coeff[sc->idx[pos] - 1] : 0, above = py > 0 ? coeff[sc->idx[pos] - w] : 0;
      const int numPos = (left != 0) + (above != 0);
      if (numNonZero || i != 15) {
        if (--remCtxBins >= 0) code_bin(e, &c->ts_sig[numPos], v != 0); else e->bits += EP_BITS;
      }
      if (v) {
        int signCtx, pred1, mod, rem;
        if ((left == 0 && above == 0) || ((int64_t)left * above < 0)) signCtx = 0;
        else if (left >= 0 && above >= 0) signCtx = 1;
        else signCtx = 2;
        if (--remCtxBins >= 0) code_bin(e, &c->ts_sign[signCtx], v < 0); else e->bits += EP_BITS;
        numNonZero++;
        pred1 = imax(abs(left), abs(above));
        mod = abs(v) == pred1 ? 1 : (abs(v) < pred1 ? abs(v) + 1 : abs(v));
        rem = mod - 1;
        if (--remCtxBins >= 0) code_bin(e, &c->ts_lrg1[numPos], rem != 0); else e->bits += EP_BITS;
        if (rem) {
          rem -= 1;
          if (--remCtxBins >= 0) code_bin(e, &c->ts_par[0], rem & 1); else e->bits += EP_BITS;
        }
      }
    }
    for (i = 0; i < 16; i++) {                                   /* greater-than-x flags, single pass (JVET_O0619) */
      const int pos = sb * 16 + i, px = sc->x[pos], py = sc->y[pos];
      const int left = px > 0 ? coeff[sc->idx[pos] - 1] : 0, above = py > 0 ? coeff[sc->idx[pos] - w] : 0;
      const int pred1 = imax(abs(left), abs(above)), a = abs(coeff[sc->idx[pos]]);
      const int mod = a == pred1 ? 1 : (a < pred1 ? a + 1 : a);
      int cutoff = 2;
      for (k = 0; k < 4; k++) {
        if (mod >= cutoff) {
          if (--remCtxBins >= 0) code_bin(e, &c->ts_gtx[cutoff >> 1], mod >= cutoff + 2); else e->bits += EP_BITS;
        }
        cutoff += 2;
      }
    }
    for (i = 0; i < 16; i++) {                                   /* remainders */
      const int pos = sb * 16 + i, px = sc->x[pos], py = sc->y[pos];
      const int left = px > 0 ? coeff[sc->idx[pos] - 1] : 0, above = py > 0 ? coeff[sc->idx[pos] - w] : 0;
      const int pred1 = imax(abs(left), abs(above)), a = abs(coeff[sc->idx[pos]]);
      const int mod = a == pred1 ? 1 : (a < pred1 ? a + 1 : a);
      if (mod >= 10) code_rem_abs_ep(e, (unsigned)(mod - 10) >> 1, kTsRicePars[imin(abs(left) + abs(above), 31)]);
    }
  }
}

uint64_t orc_residual_bits(const int32_t* coeff, int w, int h, int mts_idx, int ts_allowed, int mts_allowed, int dep_quant,
                           const vvcb_ctx_states* states)
{
  static res_scan sc;
  static const int prefixCtx[8] = { 0, 0, 0, 3, 6, 10, 15, 21 };
  vvcb_ctx_states c = *states;
  est e = { 0 };
  uint8_t sigGroup[64], coded[64];
  int scanPosLast = -1, pos, sb, state = 0, regBins;
  const int stateTab = dep_quant ? 32040 : 0;
  build_res_scan(&sc, w, h);
  memset(sigGroup, 0, sizeof(sigGroup)); memset(coded, 0, sizeof(coded));
  for (pos = 0; pos < sc.numCoeff; pos++) if (coeff[sc.idx[pos]]) { scanPosLast = pos; sigGroup[pos >> 4] = 1; }
  /* residual_coding runs only for a coded block (cbf 1): an all-zero block costs nothing, transform skip included */
  if (scanPosLast < 0) return 0;
  mts_coding(&e, &c, mts_idx, ts_allowed, mts_allowed);
  if (mts_idx == 1) { residual_ts(&e, &c, &sc, coeff); return e.bits; }
  {                                                              /* last_sig_coeff */
    int px = sc.x[scanPosLast], py = sc.y[scanPosLast];
    const int gX = kGroupIdx[px], gY = kGroupIdx[py], lw = ilog2(w), lh = ilog2(h);
    int maxX = kGroupIdx[imin(32, w) - 1], maxY = kGroupIdx[imin(32, h) - 1], k;
    if (mts_idx > 1) { if (w == 32) maxX = kGroupIdx[15]; if (h == 32) maxY = kGroupIdx[15]; }
    for (k = 0; k < gX; k++) code_bin(&e, &c.last_x[prefixCtx[lw] + (k >> ((lw + 1) >> 2))], 1);
    if (gX < maxX) code_bin(&e, &c.last_x[prefixCtx[lw] + (gX >> ((lw + 1) >> 2))], 0);
    for (k = 0; k < gY; k++) code_bin(&e, &c.last_y[prefixCtx[lh] + (k >> ((lh + 1) >> 2))], 1);
    if (gY < maxY) code_bin(&e, &c.last_y[prefixCtx[lh] + (gY >> ((lh + 1) >> 2))], 0);
    if (gX > 3) e.bits += (uint64_t)((gX - 2) >> 1) * EP_BITS;
    if (gY > 3) e.bits += (uint64_t)((gY - 2) >> 1) * EP_BITS;
    (void)kMinInGroup;
  }
  {                                                              /* TU::getTbAreaAfterCoefZeroOut x 28 >> 4 */
    int tbW = w, tbH = h;
    if (mts_idx > 1) { tbW = w == 32 ? 16 : w; tbH = h == 32 ? 16 : h; }
    regBins = (imin(32, tbW) * imin(32, tbH) * 28) >> 4;
  }
  for (sb = scanPosLast >> 4; sb >= 0; sb--) {
    const int sbPos = sc.sbbPos[sb], sy = sbPos / sc.gw, sx = sbPos - sy * sc.gw, minSub = sb * 16;
    const int isLast = (scanPosLast >> 4) == sb;
    int firstSigPos = isLast ? scanPosLast : minSub + 15, next, inferSigPos, numNonZero = 0, remReg, firstPosMode2, i;
    unsigned signBins = 0;
    if (sigGroup[sb]) coded[sbPos] = 1;                          /* initSubblock( subSetId, sigGroupFlags[subSetId] ) */
    if (mts_idx > 1 && ((h == 32 && sy >= 4) || (w == 32 && sx >= 4))) continue;
    if (!isLast && sb != 0) {
      const int sigRight = sx + 1 < sc.gw ? coded[sbPos + 1] : 0, sigLower = sy + 1 < sc.gh ? coded[sbPos + sc.gw] : 0;
      code_bin(&e, &c.sig_sbb[sigRight | sigLower], sigGroup[sb]);
      if (!sigGroup[sb]) continue;
    }
    next = firstSigPos;
    inferSigPos = next != scanPosLast ? (sb != 0 ? minSub : -1) : next;
    remReg = regBins;
    for (; next >= minSub && remReg >= 4; next--) {
      const int32_t v = coeff[sc.idx[next]];
      const int px = sc.x[next], py = sc.y[next], diag = px + py;
      int sumAbs1, numPos, sumAbs;
      template_sums(coeff, w, h, px, py, &sumAbs1, &numPos, &sumAbs);
      if (numNonZero || next != inferSigPos) {
        const int ctxOfs = imin((sumAbs1 + 1) >> 1, 3) + (diag < 2 ? 4 : 0) + (diag < 5 ? 4 : 0);
        code_bin(&e, &c.sig[imax(0, state - 1)][ctxOfs], v != 0);
        remReg--;
      }
      if (v) {
        /* ctxOffsetAbs(): m_tmplCpDiag / m_tmplCpSum1 are the ones of this position (sigCtxIdAbs has run, or the position is the last one
         * of the TU, for which they still hold their initial -1 -> offset 0) */
        int ctxOff = 0, rem = abs(v) - 1;
        if (next != scanPosLast) ctxOff = imin(sumAbs1 - numPos, 4) + 1 + (diag == 0 ? 15 : diag < 3 ? 10 : diag < 10 ? 5 : 0);
        numNonZero++;
        signBins++;
        code_bin(&e, &c.gt1[ctxOff], rem != 0);
        remReg--;
        if (rem) {
          rem -= 1;
          code_bin(&e, &c.par[ctxOff], rem & 1);
          rem >>= 1;
          remReg--;
          code_bin(&e, &c.gt2[ctxOff], rem != 0);
          remReg--;
        }
      }
      state = (stateTab >> ((state << 2) + ((v & 1) << 1))) & 3;
    }
    firstPosMode2 = next;
    regBins = remReg;
    for (i = firstSigPos; i > firstPosMode2; i--) {              /* 2nd pass: Golomb-Rice remainders */
      const int a = abs(coeff[sc.idx[i]]);
      if (a >= 4) {
        int s1, np, sa;
        template_sums(coeff, w, h, sc.x[i], sc.y[i], &s1, &np, &sa);
        code_rem_abs_ep(&e, (unsigned)(a - 4) >> 1, kRicePars[imax(imin(sa - 20, 31), 0)]);
      }
    }
    for (i = firstPosMode2; i >= minSub; i--) {                  /* bypass-coded coefficients */
      const int32_t v = coeff[sc.idx[i]];
      const int a = abs(v);
      int s1, np, sa, sumAll, pos0;
      template_sums(coeff, w, h, sc.x[i], sc.y[i], &s1, &np, &sa);
      sumAll = imax(imin(sa, 31), 0);
      pos0 = kRicePos0[imax(0, state - 1)][sumAll];
      code_rem_abs_ep(&e, (unsigned)(a == 0 ? pos0 : (a <= pos0 ? a - 1 : a)), kRicePars[sumAll]);
      state = (stateTab >> ((state << 2) + ((a & 1) << 1))) & 3;
      if (a) signBins++;
    }
    e.bits += (uint64_t)signBins * EP_BITS;
  }
  return e.bits;
}
