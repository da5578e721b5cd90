/*
 * TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the reference's dependent quantisation (trellis-coded
 * quantisation, SURVEY.md 8a row a13): DQIntern::DepQuant::quant and Quantizer::dequantBlock of CL/DepQuant.cpp,
 * luma, flat scaling, with the compile-time switches of the reference as shipped (CL/TypeDef.h: JVET_O0094, O0052,
 * O0617, O0256, O0919 all 1).  See vvc_oracle.h for who may use it.
 *
 * Parity status: PINNED.  tests/test_oracle_dq.py feeds the coefficients and context prices recorded from the unmodified
 * reference encoder ('D' records of oracle/ref_trace_hooks.cpp) and requires the identical levels and absSum.
 */
#include <stdlib.h>
#include <string.h>
#include <limits.h>
#include "vvc_oracle.h"
#include "../vvc_intra_b200/csrc/vvc_rom_tables.h"

#define SCALE_BITS 15
#define RICEMAX 32

/* CL/DepQuant.cpp:887-893 */
static const int32_t kGoRiceBits[4][RICEMAX] = {
  { 32768,  65536,  98304, 131072, 163840, 196608, 262144, 262144, 327680, 327680, 327680, 327680, 393216, 393216, 393216, 393216, 393216, 393216, 393216, 393216, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752},
  { 65536,  65536,  98304,  98304, 131072, 131072, 163840, 163840, 196608, 196608, 229376, 229376, 294912, 294912, 294912, 294912, 360448, 360448, 360448, 360448, 360448, 360448, 360448, 360448, 425984, 425984, 425984, 425984, 425984, 425984, 425984, 425984},
  { 98304,  98304,  98304,  98304, 131072, 131072, 131072, 131072, 163840, 163840, 163840, 163840, 196608, 196608, 196608, 196608, 229376, 229376, 229376, 229376, 262144, 262144, 262144, 262144, 327680, 327680, 327680, 327680, 327680, 327680, 327680, 327680},
  {131072, 131072, 131072, 131072, 131072, 131072, 131072, 131072, 163840, 163840, 163840, 163840, 163840, 163840, 163840, 163840, 196608, 196608, 196608, 196608, 196608, 196608, 196608, 196608, 229376, 229376, 229376, 229376, 229376, 229376, 229376, 229376}
};
/* CL/Rom.cpp:628-638 */
static const uint8_t kGroupIdx[64] = { 0,1,2,3,4,4,5,5,6,6,6,6,7,7,7,7,8,8,8,8,8,8,8,8,9,9,9,9,9,9,9,9, 10,10,10,10,10,10,10,10,10,10,10,10,10,10,10,10,11,11,11,11,11,11,11,11,11,11,11,11,11,11,11,11 };
static const uint8_t kGoRicePars[32] = { 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 3, 3, 3 };
static const uint8_t kGoRicePosCoeff0[3][32] = {
  {0, 0, 0, 0, 0, 1, 2,    2, 2, 2, 2, 2, 4, 4,    4, 4, 4, 4,  4,  4,  4,  4,  4,  8,  8,  8,  8,  8,     8,  8,  8,  8},
  {1, 1, 1, 1, 2, 3, 4,    4, 4, 6, 6, 6, 8, 8,    8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 12, 16, 16,    16, 16, 16, 16},
  {1, 1, 2, 2, 2, 3, 4,    4, 4, 6, 6, 6, 8, 8,    8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 16, 16, 16,    16, 16, 16, 16} };

static int ilog2(int v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }
static int imin(int a, int b) { return a < b ? a : b; }
static int imax(int a, int b) { return a > b ? a : b; }

/* ---- scan tables of one TU shape (CL/Rom.cpp:263-365 grouped 4x4 diagonal scan; CL/DepQuant.cpp:153-432) ---- */
typedef struct { uint8_t num; uint8_t inPos[5]; } nb_sbb;
typedef struct { uint16_t maxDist, num, outPos[5]; } nb_out;
typedef struct {
  int w, h, numCoeff, numSbb, widthInSbb, heightInSbb;
  uint16_t idx[1024]; uint8_t x[1024], y[1024];      /* scanId -> raster position (stride w) and coordinates */
  uint16_t sbbPos[64];                               /* sub-block scan -> raster position in the sub-block grid */
  nb_sbb nbSbb[1024];
  nb_out nbOut[1024];
} tu_scan;

/* up-right diagonal order of a bw x bh grid: anti-diagonals from the top-left, each walked from bottom-left to top-right */
static int diag_order(int bw, int bh, uint8_t* ox, uint8_t* oy)
{
  int n = 0, d, y;
  for (d = 0; d <= bw + bh - 2; d++)
    for (y = imin(d, bh - 1); y >= imax(0, d - bw + 1); y--) { ox[n] = (uint8_t)(d - y); oy[n] = (uint8_t)y; n++; }
  return n;
}

static void build_scan(tu_scan* s, int w, int h)
{
  uint8_t gx[64], gy[64], ix[16], iy[16];
  static int raster2id[64 * 64];
  int g, i, k, scanId;
  const int nzW = imin(32, w), nzH = imin(32, h);
  memset(s, 0, sizeof(*s));
  s->w = w; s->h = h; s->widthInSbb = nzW >> 2; s->heightInSbb = nzH >> 2;
  s->numSbb = s->widthInSbb * s->heightInSbb; s->numCoeff = nzW * nzH;
  diag_order(s->widthInSbb, s->heightInSbb, gx, gy);
  diag_order(4, 4, ix, iy);
  memset(raster2id, 0, sizeof(raster2id));
  for (g = 0; g < s->numSbb; g++) {
    s->sbbPos[g] = (uint16_t)(gy[g] * s->widthInSbb + gx[g]);
    for (i = 0; i < 16; i++) {
      const int id = g * 16 + i, px = gx[g] * 4 + ix[i], py = gy[g] * 4 + iy[i];
      s->x[id] = (uint8_t)px; s->y[id] = (uint8_t)py; s->idx[id] = (uint16_t)(py * w + px);
      raster2id[py * w + px] = id;
    }
  }
  for (scanId = 0; scanId < s->numCoeff; scanId++) {
    const int px = s->x[scanId], py = s->y[scanId], rpos = s->idx[scanId], beg = scanId & ~15;
    int cand[5], in[5], out[5];
    cand[0] = px + 1 < nzW ? raster2id[rpos + 1] : 0;
    cand[1] = px + 2 < nzW ? raster2id[rpos + 2] : 0;
    cand[2] = px + 1 < nzW && py + 1 < nzH ? raster2id[rpos + 1 + w] : 0;
    cand[3] = py + 1 < nzH ? raster2id[rpos + w] : 0;
    cand[4] = py + 2 < nzH ? raster2id[rpos + 2 * w] : 0;
    for (k = 0; k < 5; k++) {
      const int present = k == 0 ? px + 1 < nzW : k == 1 ? px + 2 < nzW : k == 2 ? (px + 1 < nzW && py + 1 < nzH) : k == 3 ? py + 1 < nzH : py + 2 < nzH;
      in[k]  = present && cand[k] < beg + 16 ? cand[k] - beg : 0;
      out[k] = present && cand[k] >= beg + 16 ? cand[k] : 0;
    }
    for (;;) {                                        /* ascending, zeros (absent) skipped: CL/DepQuant.cpp:214-231 */
      int nk = -1;
      for (k = 0; k < 5; k++) if (in[k] != 0 && (nk < 0 || in[k] < in[nk])) nk = k;
      if (nk < 0) break;
      s->nbSbb[scanId].inPos[s->nbSbb[scanId].num++] = (uint8_t)in[nk];
      in[nk] = 0;
    }
    for (;;) {
      int nk = -1;
      for (k = 0; k < 5; k++) if (out[k] != 0 && (nk < 0 || out[k] < out[nk])) nk = k;
      if (nk < 0) break;
      s->nbOut[scanId].outPos[s->nbOut[scanId].num++] = (uint16_t)out[nk];
      out[nk] = 0;
    }
    s->nbOut[scanId].maxDist = scanId == 0 ? 0 : s->nbOut[scanId - 1].maxDist;
    for (k = 0; k < s->nbOut[scanId].num; k++)
      if (s->nbOut[scanId].outPos[k] > s->nbOut[scanId].maxDist) s->nbOut[scanId].maxDist = s->nbOut[scanId].outPos[k];
  }
  for (scanId = 0; scanId < s->numCoeff; scanId++) {    /* "make it relative", :277-288 */
    const int beg = scanId & ~15;
    for (k = 0; k < s->nbOut[scanId].num; k++) s->nbOut[scanId].outPos[k] = (uint16_t)(s->nbOut[scanId].outPos[k] - beg);
    s->nbOut[scanId].maxDist = (uint16_t)(s->nbOut[scanId].maxDist - scanId);
  }
}

/* ---- rate tables (RateEstimator, CL/DepQuant.cpp:479-629) ---- */
typedef struct {
  int32_t lastBitsX[32], lastBitsY[32];
  int32_t sigSbb[2][2], sig[3][12][2], gtx[21][6];
} dq_rate;

static void init_rates(dq_rate* r, const vvcb_dq_rates* c, int w, int h, int cbfDeltaBits)
{
  static const unsigned prefixCtx[] = { 0, 0, 0, 3, 6, 10, 15, 21 };
  int xy, i, k;
  for (i = 0; i < 2; i++) for (k = 0; k < 2; k++) r->sigSbb[i][k] = (int32_t)c->sig_sbb[i][k];
  for (xy = 0; xy < 3; xy++) for (i = 0; i < 12; i++) for (k = 0; k < 2; k++) r->sig[xy][i][k] = (int32_t)c->sig[xy][i][k];
  for (i = 0; i < 21; i++) {                          /* xSetGtxFlagBits :597-629 */
    const int32_t par0 = (1 << SCALE_BITS) + (int32_t)c->par[i][0], par1 = (1 << SCALE_BITS) + (int32_t)c->par[i][1];
    r->gtx[i][0] = 0;
    r->gtx[i][1] = (int32_t)c->gt1[i][0] + (1 << SCALE_BITS);
    r->gtx[i][2] = (int32_t)c->gt1[i][1] + par0 + (int32_t)c->gt2[i][0];
    r->gtx[i][3] = (int32_t)c->gt1[i][1] + par1 + (int32_t)c->gt2[i][0];
    r->gtx[i][4] = (int32_t)c->gt1[i][1] + par0 + (int32_t)c->gt2[i][1];
    r->gtx[i][5] = (int32_t)c->gt1[i][1] + par1 + (int32_t)c->gt2[i][1];
  }
  for (xy = 0; xy < 2; xy++) {                        /* xSetLastCoeffOffset :541-567 */
    const int32_t bitOffset = xy ? cbfDeltaBits : 0;
    int32_t* lastBits = xy ? r->lastBitsY : r->lastBitsX;
    const int size = xy ? h : w, log2Size = ilog2(size);
    const uint32_t (*ctx)[2] = xy ? c->last_y : c->last_x;
    const unsigned lastShift = (unsigned)(log2Size + 1) >> 2, lastOffset = prefixCtx[log2Size];
    uint32_t sumFBits = 0, ctxBits[14];
    const unsigned maxCtxId = kGroupIdx[imin(32, size) - 1];
    unsigned ctxId;
    for (ctxId = 0; ctxId < maxCtxId; ctxId++) {
      const uint32_t* b = ctx[lastOffset + (ctxId >> lastShift)];
      ctxBits[ctxId] = sumFBits + b[0] + (ctxId > 3 ? ((ctxId - 2) >> 1) << SCALE_BITS : 0) + (uint32_t)bitOffset;
      sumFBits += b[1];
    }
    ctxBits[maxCtxId] = sumFBits + (maxCtxId > 3 ? ((maxCtxId - 2) >> 1) << SCALE_BITS : 0) + (uint32_t)bitOffset;
    for (i = 0; i < imin(32, size); i++) lastBits[i] = (int32_t)ctxBits[kGroupIdx[i]];
  }
}

/* ---- Quantizer (CL/DepQuant.cpp:654-844) ---- */
typedef struct {
  int qShift; int64_t qAdd, qScale; int maxQIdx, thresLast;
  int distShift; int64_t distAdd, distStepAdd, distOrgFact;
} dq_quant;

static int ceil_log2_u64(uint64_t x)                  /* :680-693 */
{
  int y = (x & (x - 1)) == 0 ? 0 : 1, n = 0;
  while (x > 1) { x >>= 1; n++; }
  return y + n;
}

static int transform_shift(int bd, int w, int h) { return 15 - bd - ((ilog2(w) + ilog2(h)) >> 1); }

static void init_quant(dq_quant* q, int bd, int w, int h, int qp, double lambda)
{
  const int qpDQ = qp + 1, qpPer = qpDQ / 6, qpRem = qpDQ - 6 * qpPer;
  const int nomTransformShift = transform_shift(bd, w, h);
  const int sqrt2 = (ilog2(w) + ilog2(h)) & 1;       /* TU::needsSqrt2Scale, no transform skip here */
  const int transformShift = nomTransformShift + (sqrt2 ? -1 : 0);
  const int invShift = 6 + 1 - qpPer - transformShift;
  int qIdxBD, nomDShift, dfShift;
  double qScale2, nomDistFactor;
  int64_t pow2dfShift;
  q->qShift = 14 - 1 + qpPer + transformShift;
  q->qAdd = -(((int64_t)3 << q->qShift) >> 1);
  q->qScale = kQuantScales[(sqrt2 ? 6 : 0) + qpRem];
  qIdxBD = imin(15 + 1, 8 * (int)sizeof(int32_t) + invShift - 6 - 1);
  q->maxQIdx = (1 << (qIdxBD - 1)) - 4;
  q->thresLast = (int)((int64_t)4 << q->qShift);
  nomDShift = SCALE_BITS - 2 * (nomTransformShift + 0) + q->qShift + (sqrt2 ? 1 : 0);   /* DISTORTION_PRECISION_ADJUSTMENT == 0 */
  qScale2 = (double)(q->qScale * q->qScale);
  nomDistFactor = nomDShift < 0 ? 1.0 / ((double)((int64_t)1 << (-nomDShift)) * qScale2 * lambda)
                                : (double)((int64_t)1 << nomDShift) / (qScale2 * lambda);
  pow2dfShift = (int64_t)(nomDistFactor * qScale2) + 1;
  dfShift = ceil_log2_u64((uint64_t)pow2dfShift);
  q->distShift = 62 + q->qShift - 2 * 15 - dfShift;
  q->distAdd = ((int64_t)1 << q->distShift) >> 1;
  /* distShift + qShift reaches 64..73 on 4x4 blocks at QP >= 48.  The reference's shift is then undefined in C++; x86 masks the count
     to its low six bits, which is written out here.  The device shift gives 0 instead; both round f * 2^(count - 64) + .5 down to 0 as
     long as that product stays below .5 (tests/test_tu_range_limits.py checks it over the QP range). */
  q->distStepAdd = (int64_t)(nomDistFactor * (double)((int64_t)1 << ((q->distShift + q->qShift) & 63)) + .5);
  q->distOrgFact = (int64_t)(nomDistFactor * (double)((int64_t)1 << (q->distShift + 1)) + .5);
}

typedef struct { int absLevel; int64_t deltaDist; } pq_data;

static void pre_quant(const dq_quant* q, int absCoeff, pq_data* pq)     /* :812-843 */
{
  const int64_t scaledOrg = (int64_t)absCoeff * q->qScale;
  int qIdx = imax(1, imin(q->maxQIdx, (int)((scaledOrg + q->qAdd) >> q->qShift)));
  int64_t scaledAdd = qIdx * q->distStepAdd - scaledOrg * q->distOrgFact;
  int k;
  for (k = 0; k < 4; k++) {
    pq_data* p = &pq[qIdx & 3];
    p->deltaDist = (scaledAdd * qIdx + q->distAdd) >> q->distShift;
    p->absLevel = (++qIdx) >> 1;
    scaledAdd += q->distStepAdd;
  }
}

/* ---- trellis ---- */
typedef struct { int64_t rdCost; int absLevel, prevId; } dq_decision;

typedef struct {
  int64_t  rdCost;
  uint16_t ctxInit[24];             /* m_absLevelsAndCtxInit: bytes 0..15 levels of the sub-block, words 8..23 template init */
  int      numSigSbb, remRegBins, refSbbCtxId;
  int32_t  sbbBits[2], sigBits[2], coefBits[6];
  int      goRicePar, goRiceZero, stateId;
} dq_state;

typedef struct {
  const tu_scan* scan; const dq_rate* rate; dq_quant quant;
  dq_state all[12], start;
  dq_state *curr, *prev, *skip;
  uint8_t mem[8 * (1024 + 64)];     /* CommonCtx::m_memory */
  uint8_t *sbbFlags[8], *levels[8]; /* m_allSbbCtx */
  int currSet, prevSet;             /* m_currSbbCtx / m_prevSbbCtx: 0 or 4 */
  int effWidth, effHeight;
  dq_decision trellis[1024][8];
} dq_ctx;

static const int32_t* sig_table(const dq_ctx* c, int stateId, int ctxId) { return c->rate->sig[imax(stateId - 1, 0)][ctxId]; }

static void state_init(dq_ctx* c, dq_state* s, int id)     /* State::init :913-923 */
{
  s->rdCost = INT64_MAX >> 1;
  s->numSigSbb = 0; s->remRegBins = 4; s->refSbbCtxId = -1;
  memcpy(s->sigBits, sig_table(c, id, 0), sizeof(s->sigBits));
  memcpy(s->coefBits, c->rate->gtx[0], sizeof(s->coefBits));
  s->goRicePar = 0; s->goRiceZero = 0; s->stateId = id;
  s->sbbBits[0] = s->sbbBits[1] = 0;
  memset(s->ctxInit, 0, sizeof(s->ctxInit));
}

static void consider(dq_decision* d, int64_t cost, int level, int prevId) { if (cost < d->rdCost) { d->rdCost = cost; d->absLevel = level; d->prevId = prevId; } }

static int64_t level_bits(const dq_state* s, int absLevel)     /* the regular-bin branch of :977-990 */
{
  if (absLevel < 4) return s->coefBits[absLevel];
  {
    const unsigned value = (unsigned)(absLevel - 4) >> 1;
    return s->coefBits[absLevel - (int)(value << 1)] + kGoRiceBits[s->goRicePar][value < RICEMAX ? value : RICEMAX - 1];
  }
}

/* State::checkRdCosts :924-1049 (JVET_O0094 on: no zero-out branch inside) */
static void check_rd_costs(const dq_state* s, int spt, const pq_data* A, const pq_data* B, dq_decision* dA, dq_decision* dB)
{
  const int32_t* rice = kGoRiceBits[s->goRicePar];
  int64_t cA = s->rdCost + A->deltaDist, cB = s->rdCost + B->deltaDist, cZ = s->rdCost;
  if (s->remRegBins >= 4) {
    cA += level_bits(s, A->absLevel);
    cB += level_bits(s, B->absLevel);
    if (spt == 0)      { cA += s->sigBits[1]; cB += s->sigBits[1]; cZ += s->sigBits[0]; }
    else if (spt == 1) { cA += s->sbbBits[1] + s->sigBits[1]; cB += s->sbbBits[1] + s->sigBits[1]; cZ += s->sbbBits[1] + s->sigBits[0]; }
    else if (s->numSigSbb) { cA += s->sigBits[1]; cB += s->sigBits[1]; cZ += s->sigBits[0]; }
    else cZ = dA->rdCost;
  } else {
    cA += (1 << SCALE_BITS) + rice[A->absLevel <= s->goRiceZero ? A->absLevel - 1 : (A->absLevel < RICEMAX ? A->absLevel : RICEMAX - 1)];
    cB += (1 << SCALE_BITS) + rice[B->absLevel <= s->goRiceZero ? B->absLevel - 1 : (B->absLevel < RICEMAX ? B->absLevel : RICEMAX - 1)];
    cZ += rice[s->goRiceZero];
  }
  consider(dA, cA, A->absLevel, s->stateId);
  consider(dA, cZ, 0, s->stateId);
  consider(dB, cB, B->absLevel, s->stateId);
}

static int scan_spt(const tu_scan* t, int scanIdx)       /* xSetScanInfo :393-397; 0 ISCSBB, 1 SOCSBB, 2 EOCSBB */
{
  const int inside = scanIdx & 15;
  if (inside == 15 && scanIdx > 16 && scanIdx < t->numCoeff - 1) return 1;
  if (inside == 0 && scanIdx > 0 && scanIdx < t->numCoeff - 16) return 2;
  return 0;
}

static void ctx_offsets_next(const tu_scan* t, int scanIdx, int* sigOff, int* gtxOff)   /* :400-425, luma */
{
  const int diag = t->x[scanIdx - 1] + t->y[scanIdx - 1];
  *sigOff = diag < 2 ? 8 : diag < 5 ? 4 : 0;
  *gtxOff = diag < 1 ? 16 : diag < 3 ? 11 : diag < 10 ? 6 : 1;
}

/* State::updateState<numIPos> :1109-1273 */
static void update_state(dq_ctx* c, dq_state* s, int scanIdx, const dq_decision* dec)
{
  const tu_scan* t = c->scan;
  uint8_t* levels = (uint8_t*)s->ctxInit;
  const nb_sbb* nb = &t->nbSbb[scanIdx - 1];
  const int nextInside = (scanIdx - 1) & 15;
  int sigOff, gtxOff, k;
  s->rdCost = dec->rdCost;
  if (dec->prevId <= -2) return;
  if (dec->prevId >= 0) {
    const dq_state* p = &c->prev[dec->prevId];
    s->numSigSbb = p->numSigSbb + !!dec->absLevel;
    s->refSbbCtxId = p->refSbbCtxId;
    memcpy(s->sbbBits, p->sbbBits, sizeof(s->sbbBits));
    s->remRegBins = p->remRegBins - 1;
    s->goRicePar = p->goRicePar;
    if (s->remRegBins >= 4) s->remRegBins -= dec->absLevel < 2 ? dec->absLevel : 3;
    memcpy(s->ctxInit, p->ctxInit, 48);
  } else {
    s->numSigSbb = 1; s->refSbbCtxId = -1;
    s->remRegBins = (c->effWidth * c->effHeight * 28) / 16 - (dec->absLevel < 2 ? dec->absLevel : 3);
    memset(s->ctxInit, 0, 48);
  }
  levels[scanIdx & 15] = (uint8_t)imin(255, dec->absLevel);
  ctx_offsets_next(t, scanIdx, &sigOff, &gtxOff);
  if (s->remRegBins >= 4) {
    const int tinit = s->ctxInit[8 + nextInside];
    int sumAbs1 = (tinit >> 3) & 31, sumNum = tinit & 7, sumAbs = tinit >> 8, sumGt1, sumAll;
    for (k = 0; k < nb->num; k++) {
      const int v = levels[nb->inPos[k]];
      sumAbs1 += imin(4 + (v & 1), v); sumNum += !!v; sumAbs += v;
    }
    sumGt1 = sumAbs1 - sumNum;
    memcpy(s->sigBits, sig_table(c, s->stateId, sigOff + imin((sumAbs1 + 1) >> 1, 3)), sizeof(s->sigBits));
    memcpy(s->coefBits, c->rate->gtx[gtxOff + (sumGt1 < 4 ? sumGt1 : 4)], sizeof(s->coefBits));
    sumAll = imax(imin(31, sumAbs - 4 * 5), 0);
    s->goRicePar = kGoRicePars[sumAll];
  } else {
    int sumAbs = s->ctxInit[8 + nextInside] >> 8;
    for (k = 0; k < nb->num; k++) sumAbs += levels[nb->inPos[k]];
    sumAbs = imin(31, sumAbs);
    s->goRicePar = kGoRicePars[sumAbs];
    s->goRiceZero = kGoRicePosCoeff0[imax(0, s->stateId - 1)][sumAbs];
  }
}

/* CommonCtx::update :1317-1397 */
static void common_update(dq_ctx* c, int scanIdx, const dq_state* prevState, dq_state* cur)
{
  const tu_scan* t = c->scan;
  uint8_t* sbbFlags = c->sbbFlags[c->currSet + cur->stateId];
  uint8_t* levels = c->levels[c->currSet + cur->stateId];
  const int setCpSize = t->nbOut[scanIdx - 1].maxDist;
  const int sbbPos = t->sbbPos[scanIdx >> 4];
  int nextSbbRight = 0, nextSbbBelow = 0, sigNSbb, id;
  uint16_t templ[16];
  const int scanBeg = scanIdx - 16;
  if (prevState && prevState->refSbbCtxId >= 0) {
    memcpy(sbbFlags, c->sbbFlags[c->prevSet + prevState->refSbbCtxId], t->numSbb);
    memcpy(levels + scanIdx, c->levels[c->prevSet + prevState->refSbbCtxId] + scanIdx, setCpSize);
  } else {
    memset(sbbFlags, 0, t->numSbb);
    memset(levels + scanIdx, 0, setCpSize);
  }
  sbbFlags[sbbPos] = !!cur->numSigSbb;
  memcpy(levels + scanIdx, cur->ctxInit, 16);
  {                                                   /* xSetScanInfo :426-433 */
    const int nextSbbPos = t->sbbPos[(scanIdx - 1) >> 4];
    const int ny = nextSbbPos / t->widthInSbb, nx = nextSbbPos - ny * t->widthInSbb;
    nextSbbRight = nx < t->widthInSbb - 1 ? nextSbbPos + 1 : 0;
    nextSbbBelow = ny < t->heightInSbb - 1 ? nextSbbPos + t->widthInSbb : 0;
  }
  sigNSbb = ((nextSbbRight ? sbbFlags[nextSbbRight] : 0) || (nextSbbBelow ? sbbFlags[nextSbbBelow] : 0)) ? 1 : 0;
  cur->numSigSbb = 0;
  if (prevState) cur->remRegBins = prevState->remRegBins;
  else           cur->remRegBins = (c->effWidth * c->effHeight * 28) / 16;
  cur->goRicePar = 0;
  cur->refSbbCtxId = cur->stateId;
  memcpy(cur->sbbBits, c->rate->sigSbb[sigNSbb], sizeof(cur->sbbBits));
  for (id = 0; id < 16; id++) {
    const nb_out* nb = &t->nbOut[scanBeg + id];
    const uint8_t* absLevels = levels + scanBeg;
    if (nb->num) {
      int sumAbs = 0, sumAbs1 = 0, sumNum = 0, k;
      for (k = 0; k < nb->num; k++) {
        const int v = absLevels[nb->outPos[k]];
        sumAbs += v; sumAbs1 += imin(4 + (v & 1), v); sumNum += !!v;
      }
      templ[id] = (uint16_t)(sumNum + (sumAbs1 << 3) + (imin(127, sumAbs) << 8));
    } else templ[id] = 0;
  }
  memset(cur->ctxInit, 0, 16);
  memcpy(cur->ctxInit + 8, templ, 32);
}

/* State::updateStateEOS :1275-1315 */
static void update_state_eos(dq_ctx* c, dq_state* s, int scanIdx, const dq_decision* dec)
{
  const dq_state* p = NULL;
  int sigOff, gtxOff, tinit, sumNum, sumAbs1, sumGt1;
  s->rdCost = dec->rdCost;
  if (dec->prevId <= -2) return;
  if (dec->prevId >= 4) { p = &c->skip[dec->prevId - 4]; s->numSigSbb = 0; memset(s->ctxInit, 0, 16); }
  else if (dec->prevId >= 0) { p = &c->prev[dec->prevId]; s->numSigSbb = p->numSigSbb + !!dec->absLevel; memcpy(s->ctxInit, p->ctxInit, 16); }
  else { s->numSigSbb = 1; memset(s->ctxInit, 0, 16); }
  ((uint8_t*)s->ctxInit)[scanIdx & 15] = (uint8_t)imin(255, dec->absLevel);
  common_update(c, scanIdx, p, s);
  ctx_offsets_next(c->scan, scanIdx, &sigOff, &gtxOff);
  tinit = s->ctxInit[8 + ((scanIdx - 1) & 15)];
  sumNum = tinit & 7; sumAbs1 = (tinit >> 3) & 31; sumGt1 = sumAbs1 - sumNum;
  memcpy(s->sigBits, sig_table(c, s->stateId, sigOff + imin((sumAbs1 + 1) >> 1, 3)), sizeof(s->sigBits));
  memcpy(s->coefBits, c->rate->gtx[gtxOff + (sumGt1 < 4 ? sumGt1 : 4)], sizeof(s->coefBits));
}

/* DepQuant::xDecide :1455-1517 + xDecideAndUpdate :1519-1589 */
static void decide_and_update(dq_ctx* c, int absCoeff, int scanIdx, int zeroOut)
{
  static const dq_decision startDec[8] = {
    { INT64_MAX >> 2, -1, -2 }, { INT64_MAX >> 2, -1, -2 }, { INT64_MAX >> 2, -1, -2 }, { INT64_MAX >> 2, -1, -2 },
    { INT64_MAX >> 2, 0, 4 }, { INT64_MAX >> 2, 0, 5 }, { INT64_MAX >> 2, 0, 6 }, { INT64_MAX >> 2, 0, 7 } };
  dq_decision* dec = c->trellis[scanIdx];
  const int spt = scan_spt(c->scan, scanIdx), eosbb = (scanIdx & 15) == 0;
  dq_state* tmp = c->prev; c->prev = c->curr; c->curr = tmp;
  int k;
  memcpy(dec, startDec, sizeof(startDec));
  if (zeroOut) {
    if (spt == 2)
      for (k = 0; k < 4; k++) { dec[k].rdCost = c->skip[k].rdCost + c->skip[k].sbbBits[0]; dec[k].absLevel = 0; dec[k].prevId = 4 + k; }
  } else {
    pq_data pq[4];
    const int lastOffset = c->rate->lastBitsX[c->scan->x[scanIdx]] + c->rate->lastBitsY[c->scan->y[scanIdx]];
    pre_quant(&c->quant, absCoeff, pq);
    check_rd_costs(&c->prev[0], spt, &pq[0], &pq[2], &dec[0], &dec[2]);
    check_rd_costs(&c->prev[1], spt, &pq[0], &pq[2], &dec[2], &dec[0]);
    check_rd_costs(&c->prev[2], spt, &pq[3], &pq[1], &dec[1], &dec[3]);
    check_rd_costs(&c->prev[3], spt, &pq[3], &pq[1], &dec[3], &dec[1]);
    if (spt == 2)
      for (k = 0; k < 4; k++) consider(&dec[k], c->skip[k].rdCost + c->skip[k].sbbBits[0], 0, 4 + k);
    consider(&dec[0], pq[0].deltaDist + lastOffset + level_bits(&c->start, pq[0].absLevel), pq[0].absLevel, -1);   /* checkRdCostStart */
    consider(&dec[2], pq[2].deltaDist + lastOffset + level_bits(&c->start, pq[2].absLevel), pq[2].absLevel, -1);
  }
  if (scanIdx) {
    if (eosbb) {
      const int sw = c->currSet; c->currSet = c->prevSet; c->prevSet = sw;      /* m_commonCtx.swap() */
      for (k = 0; k < 4; k++) update_state_eos(c, &c->curr[k], scanIdx, &dec[k]);
      memcpy(dec + 4, dec, 4 * sizeof(dq_decision));
    } else if (!zeroOut) {
      for (k = 0; k < 4; k++) update_state(c, &c->curr[k], scanIdx, &dec[k]);
    }
    if (spt == 1) { tmp = c->prev; c->prev = c->skip; c->skip = tmp; }
  }
}

/* DQIntern::DepQuant::quant :1592-1731.  qp = QpParam::Qp of the block (the +1 of dependent quantisation is applied here). */
int orc_dep_quant(const int32_t* coeff, int w, int h, int bd, int mts_idx, int lfnst_idx, int qp, double lambda,
                  const vvcb_dq_rates* rates, int cbf_delta_bits, int32_t* level)
{
  static tu_scan scan;                 /* checker: single-threaded use */
  static dq_rate rate;
  static dq_ctx ctx;
  dq_ctx* c = &ctx;
  int absSum = 0, zeroOut = 0, zeroOutforThres, effW = w, effH = h, firstTestPos, k, scanIdx, thres;
  dq_decision decision = { INT64_MAX, -1, -2 };
  int64_t minPathCost = 0;
  memset(level, 0, sizeof(int32_t) * w * h);
  build_scan(&scan, w, h);
  c->scan = &scan; c->rate = &rate;
  init_quant(&c->quant, bd, w, h, qp, lambda);
  if (mts_idx > 1) {
    effH = h == 32 ? 16 : h; effW = w == 32 ? 16 : w;
    zeroOut = effH < h || effW < w;
  }
  zeroOutforThres = zeroOut || 32 < h || 32 < w;
  firstTestPos = w * h - 1;
  if (lfnst_idx > 0) firstTestPos = ((w == 4 && h == 4) || (w == 8 && h == 8)) ? 7 : 15;
  thres = c->quant.thresLast / (4 * (int)c->quant.qScale);
  for (; firstTestPos >= 0; firstTestPos--) {
    /* positions beyond the 32x32 low-frequency region carry the scan's filler entry (w-1, h-1), CL/Rom.cpp:339-347 */
    const int px = firstTestPos < scan.numCoeff ? scan.x[firstTestPos] : w - 1, py = firstTestPos < scan.numCoeff ? scan.y[firstTestPos] : h - 1;
    if (zeroOutforThres && (px >= ((w == 32 && zeroOut) ? 16 : 32) || py >= ((h == 32 && zeroOut) ? 16 : 32))) continue;
    if (abs(coeff[py * w + px]) > thres) break;
  }
  if (firstTestPos < 0) return 0;

  init_rates(&rate, rates, w, h, cbf_delta_bits);
  for (k = 0; k < 8; k++) { c->sbbFlags[k] = c->mem + k * (scan.numSbb + scan.numCoeff); c->levels[k] = c->sbbFlags[k] + scan.numSbb; }
  c->currSet = 0; c->prevSet = 4;
  c->curr = c->all; c->prev = c->all + 4; c->skip = c->all + 8;
  for (k = 0; k < 12; k++) state_init(c, &c->all[k], k & 3);
  state_init(c, &c->start, 0);
  c->effWidth = imin(32, effW); c->effHeight = imin(32, effH);

  for (scanIdx = firstTestPos; scanIdx >= 0; scanIdx--)
    decide_and_update(c, abs(coeff[scan.idx[scanIdx]]), scanIdx, zeroOut && (scan.x[scanIdx] >= effW || scan.y[scanIdx] >= effH));

  for (k = 0; k < 4; k++)
    if (c->trellis[0][k].rdCost < minPathCost) { decision.prevId = k; minPathCost = c->trellis[0][k].rdCost; }
  for (scanIdx = 0; decision.prevId >= 0; scanIdx++) {
    decision = c->trellis[scanIdx][decision.prevId];
    level[scan.idx[scanIdx]] = coeff[scan.idx[scanIdx]] < 0 ? -decision.absLevel : decision.absLevel;
    absSum += decision.absLevel;
  }
  return absSum;
}

/* Quantizer::dequantBlock :741-810 (flat scaling) */
void orc_dep_dequant(const int32_t* level, int w, int h, int bd, int qp, int32_t* coeff)
{
  static tu_scan scan;
  const int qpDQ = qp + 1, qpPer = qpDQ / 6, qpRem = qpDQ - 6 * qpPer;
  const int sqrt2 = (ilog2(w) + ilog2(h)) & 1;
  const int transformShift = transform_shift(bd, w, h) + (sqrt2 ? -1 : 0);
  const int shift = 6 + 1 - qpPer - transformShift;
  int invQScale = kInvQuantScales[(sqrt2 ? 6 : 0) + qpRem];
  const int add = shift < 0 ? 0 : ((1 << shift) >> 1);
  int last = -1, scanIdx, state = 0;
  build_scan(&scan, w, h);
  memset(coeff, 0, sizeof(int32_t) * w * h);
  for (scanIdx = scan.numCoeff - 1; scanIdx >= 0; scanIdx--) if (level[scan.idx[scanIdx]]) { last = scanIdx; break; }
  if (last < 0) return;
  for (scanIdx = last; scanIdx >= 0; scanIdx--) {
    const int lv = level[scan.idx[scanIdx]];
    if (lv) {
      int qIdx;
      int64_t nom;
      if (shift < 0 && scanIdx == last) invQScale <<= -shift;
      qIdx = (lv << 1) + (lv > 0 ? -(state >> 1) : (state >> 1));
      nom = ((int64_t)qIdx * (int64_t)invQScale + add) >> (shift < 0 ? 0 : shift);
      coeff[scan.idx[scanIdx]] = (int32_t)(nom < -32768 ? -32768 : (nom > 32767 ? 32767 : nom));
    }
    state = (32040 >> ((state << 2) + ((lv & 1) << 1))) & 3;
  }
}
