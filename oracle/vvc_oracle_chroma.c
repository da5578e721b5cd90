/*
 * TEST INFRASTRUCTURE -- CPU restatement ("oracle") of the prediction and distortion part of the chroma intra search,
 * IntraSearch::estIntraPredChromaQT (EL/IntraSearch.cpp:1382), for 4:2:0 with sps_cclm_colocated_chroma_flag = 0.
 * See vvc_oracle.h for the rules on who may use it.
 *
 * Parity status: UNPINNED.  Every rule is restated from H.266 and the reference lines cited at each function; nothing
 * here has been compared with the reference encoder's own chroma output.  The distortions reuse the pinned orc_sad / orc_satd.
 */
#include <stdlib.h>
#include <string.h>
#include "vvc_oracle.h"
#include "vvc_oracle_chroma.h"

#define CMAX 32

static int ilog2c(int v) { int r = 0; while (v > 1) { v >>= 1; r++; } return r; }
static int iminc(int a, int b) { return a < b ? a : b; }
static int imaxc(int a, int b) { return a > b ? a : b; }
static int clipc(int v, int maxv) { return v < 0 ? 0 : (v > maxv ? maxv : v); }
/* floorLog2 of the reference (CL/CommonDef.h): -1 for 0 */
static int floor_log2(int v) { return v <= 0 ? -1 : ilog2c(v); }

/* IntraPrediction::xFillReferenceSamples (CL/IntraPrediction.cpp:1215-1468) for a chroma block, reference line 0.  The unit of the
 * availability walk is pcv.minCUWidth >> scaleX = 2 chroma samples in 4:2:0; unavailable samples are padded from the nearest
 * earlier sample on the walk bottom-left -> corner -> top-right, those before the first available one from it, and with nothing
 * available every sample is 1 << (bd - 1) -- the luma walk of orc_ref_fill with a unit of 2.  top[0] == left[0] is the corner; 2w + 1 / 2h + 1 samples. */
void orc_chroma_ref_fill(const int16_t* reco, int stride, int x, int y, int w, int h, int bd,
                         int avail_al, int n_above, int n_above_right, int n_left, int n_below_left, int16_t* top, int16_t* left)
{
  const int nTop = 2 * w + 1, nLeft = 2 * h + 1, len = (nLeft - 1) + nTop;
  int16_t val[4 * CMAX + 2];
  uint8_t ok[4 * CMAX + 2];
  int i, first;
  for (i = 0; i < len; i++) {
    const int isLeft = i < nLeft - 1;
    const int k = isLeft ? nLeft - 1 - i : i - (nLeft - 1);
    int avail;
    if (k == 0) avail = avail_al;
    else {
      const int unit = (k - 1) >> 1;
      if (isLeft) avail = unit < (h >> 1) ? unit < n_left : unit - (h >> 1) < n_below_left;
      else        avail = unit < (w >> 1) ? unit < n_above : unit - (w >> 1) < n_above_right;
    }
    ok[i] = (uint8_t)avail;
    val[i] = avail ? (isLeft ? reco[(y - 1 + k) * stride + x - 1] : reco[(y - 1) * stride + x - 1 + k]) : 0;
  }
  for (first = 0; first < len && !ok[first]; first++) {}
  if (first == len) for (i = 0; i < len; i++) val[i] = (int16_t)(1 << (bd - 1));
  else {
    for (i = 0; i < first; i++) val[i] = val[first];
    for (i = first + 1; i < len; i++) if (!ok[i]) val[i] = val[i - 1];
  }
  for (i = 0; i < len; i++) {
    if (i < nLeft - 1) left[nLeft - 1 - i] = val[i];
    else               top[i - (nLeft - 1)] = val[i];
  }
  left[0] = top[0];
}

/* IntraPrediction::initPredIntraParams (CL/IntraPrediction.cpp:487-618) for a chroma block: wide-angle remap, intraPredAngle, invAngle,
 * PDPC (blocks of at least 4x4) and its scale from the block's own shape, as for luma; the smoothing branch is taken for luma only
 * ("!isLuma( chType )"), so refFilterFlag and interpolationFlag stay false. */
void orc_chroma_ipa_init(int w, int h, int mode, orc_ipa* p)
{
  orc_ipa_init(w, h, mode, 0, 0, p);
  p->ref_filter = 0;
  p->interp = 0;
}

/* IntraPrediction::xPredIntraAng (CL/IntraPrediction.cpp:633-935) for a chroma block.  Main reference with the projected side for
 * negative angles (:654-673) or extended by replicating its last sample twice for positive ones (:702-726); each row at
 * deltaPos = (y + 1) * intraPredAngle; a fractional position uses the 2-tap linear filter of the non-luma branch:
 * ((32 - deltaFract) * refMain[x + deltaInt + 1] + deltaFract * refMain[x + deltaInt + 2] + 16) >> 5, an integer one copies
 * refMain[x + deltaInt + 1]; PDPC of HOR / VER (clipped) and of positive angles as for luma. */
void orc_chroma_pred_angular(const int16_t* top, const int16_t* left, int w, int h, int bd, const orc_ipa* p, int16_t* pred)
{
  const int16_t* mainSrc = p->is_ver ? top : left;
  const int16_t* sideSrc = p->is_ver ? left : top;
  const int mw = p->is_ver ? w : h, mh = p->is_ver ? h : w, angle = p->angle, maxv = (1 << bd) - 1;
  int16_t mainBuf[4 * CMAX + 8], refSide[2 * CMAX + 4];
  int16_t* refMain = mainBuf + CMAX;
  int i, r, c;
  if (angle < 0) {
    for (i = 0; i <= mw + 1; i++) refMain[i] = mainSrc[i];
    for (i = 0; i <= mh + 1; i++) refSide[i] = sideSrc[i];
    for (i = -mh; i <= -1; i++) refMain[i] = refSide[iminc((-i * p->inv_angle + 256) >> 9, mh)];
  } else {
    for (i = 0; i <= 2 * mw; i++) refMain[i] = mainSrc[i];
    for (i = 0; i <= 2 * mh; i++) refSide[i] = sideSrc[i];
    for (i = 1; i <= 2; i++) refMain[2 * mw + i] = refMain[2 * mw];
  }
  for (r = 0; r < mh; r++) {
    int line[CMAX];
    if (angle == 0) {
      for (c = 0; c < mw; c++) line[c] = refMain[c + 1];
      if (p->pdpc) {
        const int scale = (ilog2c(mw) + ilog2c(mh) - 2) >> 2, lim = iminc(3 << scale, mw);
        for (c = 0; c < lim; c++) {
          const int wL = 32 >> ((2 * c) >> scale);
          line[c] = clipc(line[c] + ((wL * (refSide[1 + r] - refMain[0]) + 32) >> 6), maxv);
        }
      }
    } else {
      const int pos = angle * (r + 1), dInt = pos >> 5, dFrac = pos & 31;
      for (c = 0; c < mw; c++)
        line[c] = dFrac ? ((32 - dFrac) * refMain[c + dInt + 1] + dFrac * refMain[c + dInt + 2] + 16) >> 5 : refMain[c + dInt + 1];
      if (p->pdpc) {
        const int scale = p->ang_scale, lim = iminc(3 << scale, mw);
        int acc = 256;
        for (c = 0; c < lim; c++) {
          const int wL = 32 >> ((2 * c) >> scale);
          int l;
          acc += p->inv_angle;
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

/* IntraPrediction::xGetLumaRecPixels (CL/IntraPrediction.cpp:1665-2150 holds it with xGetLMParameters and predIntraChromaLM), 4:2:0,
 * sps_cclm_colocated_chroma_flag = 0 (the INTRA_LT_CCLM / INTRA_L_CCLM / INTRA_T_CCLM clause of H.266, the [1 2 1; 1 2 1] / 8
 * filter).  luma points at the collocated luma sample (2x, 2y) of the chroma block.
 *   ds[j][i]   = (2 Y[2j][2i] + Y[2j][2i-1] + Y[2j][2i+1] + 2 Y[2j+1][2i] + Y[2j+1][2i-1] + Y[2j+1][2i+1] + 4) >> 3
 *   ds_top[i]  = the same on luma rows -2 and -1, i < n_top
 *              = (2 Y[-1][2i] + Y[-1][2i-1] + Y[-1][2i+1] + 2) >> 2 when the block's first chroma row starts a CTU: one luma row
 *   ds_left[j] = (2 Y[2j][-2] + Y[2j][-3] + Y[2j][-1] + 2 Y[2j+1][-2] + Y[2j+1][-3] + Y[2j+1][-1] + 4) >> 3, j < n_left
 * Padding: without the left neighbours the column left of the block is replaced by its first column -- in the block (i = 0, "leftPadding")
 * and in the top neighbours (i = 0).  With them, top sample 0 reads the luma above-left corner (column -1 of rows
 * -2 / -1).  The left neighbours read only columns -3..-1 of rows 0..2 n_left - 1 and need no padding. */
void orc_cclm_luma(const int16_t* luma, int lstride, int w, int h, int avail_l, int ctu_top, int n_top, int n_left,
                   int16_t* ds, int16_t* ds_top, int16_t* ds_left)
{
  int i, j;
  for (j = 0; j < h; j++)
    for (i = 0; i < w; i++) {
      const int16_t* r0 = luma + (2 * j) * lstride;
      const int16_t* r1 = r0 + lstride;
      const int xl = 2 * i - ((i == 0 && !avail_l) ? 0 : 1);
      ds[j * w + i] = (int16_t)((2 * r0[2 * i] + r0[2 * i + 1] + r0[xl] + 2 * r1[2 * i] + r1[2 * i + 1] + r1[xl] + 4) >> 3);
    }
  for (i = 0; i < n_top; i++) {
    const int xl = 2 * i - ((i == 0 && !avail_l) ? 0 : 1);
    if (ctu_top) {
      const int16_t* r = luma - lstride;
      ds_top[i] = (int16_t)((2 * r[2 * i] + r[2 * i + 1] + r[xl] + 2) >> 2);
    } else {
      const int16_t* r0 = luma - 2 * lstride;
      const int16_t* r1 = luma - lstride;
      ds_top[i] = (int16_t)((2 * r0[2 * i] + r0[2 * i + 1] + r0[xl] + 2 * r1[2 * i] + r1[2 * i + 1] + r1[xl] + 4) >> 3);
    }
  }
  for (j = 0; j < n_left; j++) {
    const int16_t* r0 = luma + (2 * j) * lstride - 3;
    const int16_t* r1 = r0 + lstride;
    ds_left[j] = (int16_t)((2 * r0[1] + r0[2] + r0[0] + 2 * r1[1] + r1[2] + r1[0] + 4) >> 3);
  }
}

/* IntraPrediction::xGetLMParameters (CL/IntraPrediction.cpp:1665-2150; the same clause of H.266).  lm: 0 LM (67), 1 MDLM_L (68), 2 MDLM_T (69).
 * avail_t / avail_l: the whole above row / left column of the block is available; n_ar / n_bl: available above-right / below-left
 * samples (only counted when the side itself is available).  c_top / c_left: the chroma reference lines (index 0 = corner).
 *   numSampT = LM: w, MDLM_T: w + min(n_ar, h); numSampL = LM: h, MDLM_L: h + min(n_bl, w); MDLM_T ignores the left, MDLM_L the top.
 *   numIs4N = (availT && availL && LM) ? 0 : 1; startPos = numSamp >> (2 + numIs4N); pickStep = max(1, numSamp >> (1 + numIs4N));
 *   cnt = min(numSamp, (1 + numIs4N) << 1) positions per side, top ones first.
 *   Two samples in all: duplicated as {1, 0, 1, 0}.  The two smaller and two larger luma values by four compares,
 *   averaged with (a + b + 1) >> 1; then diff = maxY - minY and, for diff > 0, x = floorLog2(diff), normDiff = ((diff << 4) >> x) & 15,
 *   v = DivSigTable[normDiff] | 8, x += normDiff != 0, y = floorLog2(|diffC|) + 1, a = (diffC v + (1 << y >> 1)) >> y, k = 3 + x - y
 *   (k < 1: k = 1, a = sign(a) 15), b = minC - ((a minY) >> k); diff = 0: a = 0, k = 0, b = minC; no side at all: a = 0, k = 0,
 *   b = 1 << (bd - 1). */
void orc_cclm_params(int lm, int w, int h, int bd, int avail_t, int avail_l, int n_ar, int n_bl,
                     const int16_t* ds_top, const int16_t* ds_left, const int16_t* c_top, const int16_t* c_left, int* a, int* k, int* b)
{
  static const int DivSigTable[16] = { 0, 7, 6, 5, 5, 4, 4, 3, 3, 2, 2, 1, 1, 1, 1, 0 };
  int numT = 0, numL = 0, cntT = 0, cntL = 0, cnt, pos, i;
  int selY[4] = { 0, 0, 0, 0 }, selC[4] = { 0, 0, 0, 0 };
  int minG[2] = { 0, 2 }, maxG[2] = { 1, 3 };
  int t, minY, minC, maxY, maxC;
  if (lm == 2) { avail_l = 0; numT = w + iminc(n_ar, h); }
  else if (lm == 1) { avail_t = 0; numL = h + iminc(n_bl, w); }
  else { numT = w; numL = h; }
  {
    const int aboveIs4 = avail_l ? 0 : 1, leftIs4 = avail_t ? 0 : 1;
    if (avail_t) {
      const int start = numT >> (2 + aboveIs4), step = imaxc(1, numT >> (1 + aboveIs4));
      cntT = iminc(numT, (1 + aboveIs4) << 1);
      for (i = 0, pos = start; i < cntT; i++, pos += step) { selY[i] = ds_top[pos]; selC[i] = c_top[1 + pos]; }
    }
    if (avail_l) {
      const int start = numL >> (2 + leftIs4), step = imaxc(1, numL >> (1 + leftIs4));
      cntL = iminc(numL, (1 + leftIs4) << 1);
      for (i = 0, pos = start; i < cntL; i++, pos += step) { selY[cntT + i] = ds_left[pos]; selC[cntT + i] = c_left[1 + pos]; }
    }
  }
  cnt = cntT + cntL;
  if (!avail_t && !avail_l) { *a = 0; *k = 0; *b = 1 << (bd - 1); return; }
  if (cnt == 2) {
    selY[3] = selY[0]; selC[3] = selC[0];
    selY[2] = selY[1]; selC[2] = selC[1];
    selY[0] = selY[1]; selC[0] = selC[1];
    selY[1] = selY[3]; selC[1] = selC[3];
  }
  if (selY[minG[0]] > selY[minG[1]]) { t = minG[0]; minG[0] = minG[1]; minG[1] = t; }
  if (selY[maxG[0]] > selY[maxG[1]]) { t = maxG[0]; maxG[0] = maxG[1]; maxG[1] = t; }
  if (selY[minG[0]] > selY[maxG[1]]) {
    t = minG[0]; minG[0] = maxG[0]; maxG[0] = t;
    t = minG[1]; minG[1] = maxG[1]; maxG[1] = t;
  }
  if (selY[minG[1]] > selY[maxG[0]]) { t = minG[1]; minG[1] = maxG[0]; maxG[0] = t; }
  minY = (selY[minG[0]] + selY[minG[1]] + 1) >> 1;
  minC = (selC[minG[0]] + selC[minG[1]] + 1) >> 1;
  maxY = (selY[maxG[0]] + selY[maxG[1]] + 1) >> 1;
  maxC = (selC[maxG[0]] + selC[maxG[1]] + 1) >> 1;
  {
    const int diff = maxY - minY;
    if (diff > 0) {
      const int diffC = maxC - minC;
      int x = floor_log2(diff);
      const int normDiff = ((diff << 4) >> x) & 15;
      const int v = DivSigTable[normDiff] | 8;
      int y, aa, kk;
      x += normDiff != 0;
      y = floor_log2(abs(diffC)) + 1;
      aa = (diffC * v + (1 << y >> 1)) >> y;
      kk = 3 + x - y;
      if (kk < 1) { kk = 1; aa = aa == 0 ? 0 : (aa < 0 ? -15 : 15); }
      *a = aa; *k = kk; *b = minC - ((aa * minY) >> kk);
    } else { *a = 0; *k = 0; *b = minC; }
  }
}

/* IntraPrediction::predIntraChromaLM (CL/IntraPrediction.cpp:1665-2150): pred = Clip1(((ds a) >> k) + b) (PelBuf::linearTransform). */
void orc_cclm_pred(const int16_t* ds, int w, int h, int bd, int a, int k, int b, int16_t* pred)
{
  int i;
  for (i = 0; i < w * h; i++) pred[i] = (int16_t)clipc(((ds[i] * a) >> k) + b, (1 << bd) - 1);
}

/* PU::getIntraChromaCandModes (CL/UnitTools.cpp): PLANAR, VER, HOR, DC, LM, MDLM_L, MDLM_T, DM; the first of the four
 * regular modes that equals the DM mode becomes VDIA (66). */
void orc_chroma_cand_modes(int dm_mode, uint8_t modes[VVCB_CHROMA_CANDS])
{
  static const uint8_t base[VVCB_CHROMA_CANDS] = { 0, 50, 18, 1, VVCB_LM_CHROMA, VVCB_MDLM_L, VVCB_MDLM_T, VVCB_DM_CHROMA };
  int i;
  memcpy(modes, base, VVCB_CHROMA_CANDS);
  for (i = 0; i < 4; i++) if (modes[i] == dm_mode) { modes[i] = 66; break; }
}

/* The prediction of one chroma component under every candidate, with SAD / SATD: what estIntraPredChromaQT evaluates per candidate
 * before its transform coding (EL/IntraSearch.cpp:1382-1560).  planes[0..1]: Cb / Cr originals, planes[2..3]: Cb / Cr reconstructions
 * (stride cstride); luma: the luma reconstruction (stride lstride).  pred_out (optional): [8][2][h][w]. */
void orc_chroma_visit(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                      const vvcb_chroma_visit* v, vvcb_chroma_result* out, int16_t* pred_out)
{
  const int w = 1 << v->log2w, h = 1 << v->log2h, x = v->x, y = v->y;
  const int avail_t = v->n_above == (w >> 1), avail_l = v->n_left == (h >> 1);
  const int n_ar = avail_t ? 2 * v->n_above_right : 0, n_bl = avail_l ? 2 * v->n_below_left : 0;
  const int ctu_top = (y & ((ctu >> 1) - 1)) == 0;     /* xGetLumaRecPixels: the block's chroma y on the chroma CTU grid */
  int16_t ds[CMAX * CMAX], ds_top[2 * CMAX], ds_left[2 * CMAX];
  int16_t top[2][2 * CMAX + 1], left[2][2 * CMAX + 1], pred[CMAX * CMAX];
  int c, comp;
  memset(out, 0, sizeof(*out));
  orc_chroma_cand_modes(v->dm_mode, out->mode);
  for (comp = 0; comp < 2; comp++)
    orc_chroma_ref_fill(planes[2 + comp], cstride, x, y, w, h, bd, v->avail_al, v->n_above, v->n_above_right, v->n_left, v->n_below_left,
                        top[comp], left[comp]);
  if (v->cclm)
    orc_cclm_luma(luma + (size_t)(2 * y) * lstride + 2 * x, lstride, w, h, avail_l, ctu_top, avail_t ? w + n_ar : 0, avail_l ? h + n_bl : 0,
                  ds, ds_top, ds_left);
  for (c = 0; c < VVCB_CHROMA_CANDS; c++)
    for (comp = 0; comp < 2; comp++) {
      const int code = out->mode[c];
      const int mode = code == VVCB_DM_CHROMA ? v->dm_mode : code;
      const int16_t* org = planes[comp] + (size_t)y * cstride + x;
      if (mode >= VVCB_LM_CHROMA && mode <= VVCB_MDLM_T) {
        int a, k, b;
        if (!v->cclm) { out->sad[c][comp] = out->satd[c][comp] = VVCB_SAT_NONE; continue; }
        orc_cclm_params(mode - VVCB_LM_CHROMA, w, h, bd, avail_t, avail_l, n_ar, n_bl, ds_top, ds_left, top[comp], left[comp], &a, &k, &b);
        orc_cclm_pred(ds, w, h, bd, a, k, b, pred);
      } else {
        orc_ipa p;
        orc_chroma_ipa_init(w, h, mode, &p);
        if (mode <= 1) orc_pred_regular(top[comp], left[comp], w, h, bd, mode, &p, pred);
        else orc_chroma_pred_angular(top[comp], left[comp], w, h, bd, &p, pred);
      }
      out->sad[c][comp] = (uint32_t)orc_sad(org, cstride, pred, w, w, h);
      out->satd[c][comp] = (uint32_t)orc_satd(org, cstride, pred, w, w, h);
      if (pred_out) memcpy(pred_out + (size_t)(c * 2 + comp) * w * h, pred, sizeof(int16_t) * w * h);
    }
}

/* a batch; pred_out (optional) holds the visits' blocks one after another, 16 w h samples each */
void orc_chroma_batch(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                      const vvcb_chroma_visit* v, int n, vvcb_chroma_result* out, int16_t* pred_out)
{
  size_t off = 0;
  int i;
  for (i = 0; i < n; i++) {
    orc_chroma_visit(planes, cstride, luma, lstride, bd, ctu, v + i, out + i, pred_out ? pred_out + off : 0);
    off += (size_t)VVCB_CHROMA_CANDS * 2 << (v[i].log2w + v[i].log2h);
  }
}
