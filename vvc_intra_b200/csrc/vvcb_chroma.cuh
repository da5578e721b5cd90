// vvc_intra_b200 -- chroma intra candidates (vvcb_chroma_eval): prediction of Cb and Cr under the 8 candidates of
// PU::getIntraChromaCandModes and their SAD / SATD, 4:2:0.  Included by vvcb_api.cu and, through the CUDA-on-pthreads shim, by
// tests/host_emul/emul_chroma.cpp, emul_chroma_tu.cpp and emul_chroma_joint.cpp.
//
// One warp per visit (a chroma CU of the separate tree), warps striding over the batch:
//   1. the Cb and Cr reference lines into shared memory -- the luma padding walk (build_line_set) with a unit of 2 samples, line 0 only,
//      never smoothed -- and the block's originals;
//   2. with the LM modes enabled, the down-sampled luma of the block and of its neighbours, shared by Cb and Cr, then the (a, k, b) of
//      the three LM modes for both components; the DC values; the projected main reference of DM when its angle is negative;
//   3. the 16 evaluations (8 candidates x Cb / Cr) as lane tasks: a lane predicts one 8x8 unit (both sides >= 8) or one SATD tile (a side
//      of 4) into registers and takes residual, SAD and Walsh-Hadamard SATD with the luma tile functions; the tile follows from the
//      block's shape as xGetHADs chooses it (make_shape), the 16x8 / 8x16 tiles butterfly with the partner lane.
// Restated from H.266 and CL/IntraPrediction.cpp:487-618, 633-935, 1215-1468, 1665-2150; parity with the reference encoder's own chroma
// output is unpinned.
#pragma once
#include "vvcb_rmd.cuh"

namespace {

constexpr int kChromaWarps = 4;
constexpr int kChromaMax   = 32;           // largest chroma side evaluated
constexpr int kChromaLine  = 72;           // 2 * 32 + 1 samples + the 2 replicated ones of positive angles, rounded up to whole words

struct ChromaSmem {                        // one visit, one warp
  int16_t lines[2][2][kChromaLine];        // [0 Cb, 1 Cr][0 top / 1 left][index]: build_line_set's layout with one "set" per component
  alignas(8) int16_t org[2][kChromaMax * kChromaMax];   // the block's originals, dense w*h (residual_unit reads 4 samples at a time)
  int16_t ds[kChromaMax * kChromaMax];     // down-sampled luma of the block, dense w*h
  int16_t dsTop[2 * kChromaMax], dsLeft[2 * kChromaMax];
  alignas(4) int16_t proj[2][kChromaLine]; // DM's main reference with its projected part (build_projected_line), negative angles only
  int lm[3][2][3];                         // [LM, MDLM_L, MDLM_T][Cb, Cr]: a, k, b
  int dc[2];
};

struct ChromaParams {
  const vvcb_chroma_visit* visits;
  int n;
  vvcb_chroma_result* results;
  int16_t* predOut;                        // optional: per visit 8 x 2 blocks of w*h at predOff[visit]
  const uint32_t* predOff;
  const int16_t* orig[2];                  // Cb, Cr
  const int16_t* reco[2];
  int cstride;
  const int16_t* luma;                     // luma reconstruction
  int lstride;
  int bd, ctu;
  const Rom* rom;
};

// PU::getIntraChromaCandModes: PLANAR, VER, HOR, DC, LM, MDLM_L, MDLM_T, DM; the first regular one equal to DM becomes VDIA
__host__ __device__ __forceinline__ int chroma_cand_code(int c, int dm)
{
  const int base = c == 0 ? 0 : c == 1 ? 50 : c == 2 ? 18 : c == 3 ? 1 : VVCB_LM_CHROMA + c - 4;
  if (c < 4) {
    const int first = dm == 0 ? 0 : dm == 50 ? 1 : dm == 18 ? 2 : dm == 1 ? 3 : 4;
    if (first == c) return 66;
  }
  return base;
}

// xGetLMParameters for one LM mode (0 LM, 1 MDLM_L, 2 MDLM_T) and component
__device__ __forceinline__ void chroma_lm_params(const ChromaSmem& sm, int lm, int comp, int w, int h, int bd, bool availT, bool availL,
                                                 int nAr, int nBl, int (&out)[3])
{
  const int16_t* cTop = sm.lines[comp][0] + 1;
  const int16_t* cLeft = sm.lines[comp][1] + 1;
  int numT = w, numL = h;
  if (lm == 2) { availL = false; numT = w + vmin(nAr, h); }
  if (lm == 1) { availT = false; numL = h + vmin(nBl, w); }
  if (!availT && !availL) { out[0] = 0; out[1] = 0; out[2] = 1 << (bd - 1); return; }
  int selY[4] = { 0, 0, 0, 0 }, selC[4] = { 0, 0, 0, 0 };
  int cntT = 0, cntL = 0;
  if (availT) {
    const int is4 = availL ? 0 : 1;
    const int start = numT >> (2 + is4), step = vmax(1, numT >> (1 + is4));
    cntT = vmin(numT, (1 + is4) << 1);
    for (int i = 0; i < cntT; i++) { selY[i] = sm.dsTop[start + i * step]; selC[i] = cTop[start + i * step]; }
  }
  if (availL) {
    const int is4 = availT ? 0 : 1;
    const int start = numL >> (2 + is4), step = vmax(1, numL >> (1 + is4));
    cntL = vmin(numL, (1 + is4) << 1);
    for (int i = 0; i < cntL; i++) { selY[cntT + i] = sm.dsLeft[start + i * step]; selC[cntT + i] = cLeft[start + i * step]; }
  }
  if (cntT + cntL == 2) {
    selY[3] = selY[0]; selC[3] = selC[0]; selY[2] = selY[1]; selC[2] = selC[1];
    selY[0] = selY[1]; selC[0] = selC[1]; selY[1] = selY[3]; selC[1] = selC[3];
  }
  int mn0 = 0, mn1 = 2, mx0 = 1, mx1 = 3, t;
  if (selY[mn0] > selY[mn1]) { t = mn0; mn0 = mn1; mn1 = t; }
  if (selY[mx0] > selY[mx1]) { t = mx0; mx0 = mx1; mx1 = t; }
  if (selY[mn0] > selY[mx1]) { t = mn0; mn0 = mx0; mx0 = t; t = mn1; mn1 = mx1; mx1 = t; }
  if (selY[mn1] > selY[mx0]) { t = mn1; mn1 = mx0; mx0 = t; }
  const int minY = (selY[mn0] + selY[mn1] + 1) >> 1, minC = (selC[mn0] + selC[mn1] + 1) >> 1;
  const int maxY = (selY[mx0] + selY[mx1] + 1) >> 1, maxC = (selC[mx0] + selC[mx1] + 1) >> 1;
  const int diff = maxY - minY;
  if (diff <= 0) { out[0] = 0; out[1] = 0; out[2] = minC; return; }
  const int divSig[16] = { 0, 7, 6, 5, 5, 4, 4, 3, 3, 2, 2, 1, 1, 1, 1, 0 };
  const int diffC = maxC - minC;
  int x = vlog2(diff);
  const int normDiff = ((diff << 4) >> x) & 15;
  const int v = divSig[normDiff] | 8;
  x += normDiff != 0;
  const int y = diffC ? vlog2(vabs(diffC)) + 1 : 0;
  int a = (diffC * v + (1 << y >> 1)) >> y;
  int k = 3 + x - y;
  if (k < 1) { k = 1; a = a == 0 ? 0 : (a < 0 ? -15 : 15); }
  out[0] = a; out[1] = k; out[2] = minC - ((a * minY) >> k);
}

// one candidate of one component, as the lane tasks see it
struct ChromaCand {
  int kind;               // 0 planar, 1 DC, 2 angular, 3 LM
  int comp;
  ModeParam p;
  int a, k, b, dc;
};

// the R x C piece of the block at (x0, y0), block orientation
template <int R, int C>
__device__ __forceinline__ void chroma_predict_piece(const ChromaSmem& sm, const ChromaCand& cd, const Shape& sh, const uint32_t* filt, int maxv,
                                                     int x0, int y0, int (&q)[R][C])
{
  const int16_t* top = sm.lines[cd.comp][0];
  const int16_t* left = sm.lines[cd.comp][1];
  if (cd.kind == 3) {
#pragma unroll
    for (int i = 0; i < R; i++)
#pragma unroll
      for (int j = 0; j < C; j++) q[i][j] = clip_bd(((sm.ds[(y0 + i) * sh.w + x0 + j] * cd.a) >> cd.k) + cd.b, maxv);
  } else if (cd.kind < 2) {
    pred_planar_dc_unit<R, C>(top, left, cd.kind, cd.p.pdpc, cd.dc, sh.lw, sh.lh, x0, y0, q);
  } else if (cd.p.is_ver) {
    const int16_t* ml = cd.p.angle < 0 ? sm.proj[cd.comp] + sh.h : top;
    pred_angular_unit<R, C, true>(ml, left, cd.p, 0, sh.w, sh.h, x0, y0, filt, maxv, q);
  } else {
    int t[C][R];                                           // main/side frame of a horizontal mode: t[i][j] is block sample (y0 + j, x0 + i)
    const int16_t* ml = cd.p.angle < 0 ? sm.proj[cd.comp] + sh.w : left;
    pred_angular_unit<C, R, true>(ml, top, cd.p, 0, sh.h, sh.w, y0, x0, filt, maxv, t);
#pragma unroll
    for (int i = 0; i < R; i++)
#pragma unroll
      for (int j = 0; j < C; j++) q[i][j] = t[j][i];
  }
}

// Steps 1 and 2 for one visit, the whole warp: reference lines, originals, down-sampled luma, LM parameters, DC values, DM's projected
// main reference into sm.  Returns the block's shape; sm is complete for every lane on return.
__device__ __forceinline__ Shape chroma_visit_setup(ChromaSmem& sm, const ChromaParams& P, const Rom& rom, const vvcb_chroma_visit& cv, int lane)
{
  const Shape sh = make_shape(cv.log2w, cv.log2h);
  const int w = sh.w, h = sh.h;
  vvcb_rmd_visit lv = {};                                // the walk's view of the visit (position, size, availability)
  lv.x = cv.x; lv.y = cv.y; lv.log2w = cv.log2w; lv.log2h = cv.log2h;
  lv.avail_al = cv.avail_al; lv.n_above = cv.n_above; lv.n_above_right = cv.n_above_right; lv.n_left = cv.n_left; lv.n_below_left = cv.n_below_left;
  const bool availT = cv.n_above == (w >> 1), availL = cv.n_left == (h >> 1);
  const int nAr = availT ? 2 * cv.n_above_right : 0, nBl = availL ? 2 * cv.n_below_left : 0;
  const int dm = cv.dm_mode;
  ModeParam dmp = rom.mode[sh.lw - 2][sh.lh - 2][dm];
  __syncwarp();
  // ---- 1. reference lines and originals
#pragma unroll 1
  for (int c = 0; c < 2; c++) build_line_set<2>(sm, c, 0, lv, sh, P.reco[c], P.cstride, P.bd, lane);
  for (int i = lane; i < 2 * w * h; i += 32) {
    const int c = i >> (sh.lw + sh.lh), s = i & (w * h - 1);
    sm.org[c][s] = P.orig[c][(size_t)(cv.y + (s >> sh.lw)) * P.cstride + cv.x + (s & (w - 1))];
  }
  // ---- 2. down-sampled luma (xGetLumaRecPixels, 4:2:0, [1 2 1; 1 2 1] / 8; one row [1 2 1] / 4 above a CTU's first row)
  if (cv.cclm) {
    const int16_t* Y = P.luma + (size_t)(2 * cv.y) * P.lstride + 2 * cv.x;
    const int ls = P.lstride;
    const bool ctuTop = (cv.y & ((P.ctu >> 1) - 1)) == 0;
    const int nTop = availT ? w + vmin(nAr, h) : 0, nLeft = availL ? h + vmin(nBl, w) : 0;
    for (int i = lane; i < w * h + nTop + nLeft; i += 32) {
      int v;
      if (i < w * h + nTop) {
        const int x = i < w * h ? i & (w - 1) : i - w * h;
        const int xl = 2 * x - (x == 0 && !availL ? 0 : 1);      // no left neighbours: column -1 padded from column 0
        const int16_t* r0 = i < w * h ? Y + (size_t)(2 * (i >> sh.lw)) * ls : Y - 2 * ls;
        if (i >= w * h && ctuTop) v = (2 * r0[ls + 2 * x] + r0[ls + 2 * x + 1] + r0[ls + xl] + 2) >> 2;
        else v = (2 * r0[2 * x] + r0[2 * x + 1] + r0[xl] + 2 * r0[ls + 2 * x] + r0[ls + 2 * x + 1] + r0[ls + xl] + 4) >> 3;
        if (i < w * h) sm.ds[i] = (int16_t)v;
        else sm.dsTop[x] = (int16_t)v;
      } else {
        const int j = i - w * h - nTop;
        const int16_t* r0 = Y + (size_t)(2 * j) * ls - 3;
        sm.dsLeft[j] = (int16_t)((2 * r0[1] + r0[2] + r0[0] + 2 * r0[ls + 1] + r0[ls + 2] + r0[ls] + 4) >> 3);
      }
    }
  }
  __syncwarp();
  // LM parameters (lanes 0..5), DC values (lanes 6, 7), DM's projected main reference (every lane)
  if (cv.cclm && lane < 6) {
    int o[3];
    chroma_lm_params(sm, lane >> 1, lane & 1, w, h, P.bd, availT, availL, nAr, nBl, o);
    sm.lm[lane >> 1][lane & 1][0] = o[0]; sm.lm[lane >> 1][lane & 1][1] = o[1]; sm.lm[lane >> 1][lane & 1][2] = o[2];
  } else if (lane == 6 || lane == 7) {
    const int c = lane - 6;
    int sum = 0;
    if (w >= h) for (int i = 0; i < w; i++) sum += sm.lines[c][0][1 + i];
    if (w <= h) for (int i = 0; i < h; i++) sum += sm.lines[c][1][1 + i];
    const int denom = w == h ? 2 * w : vmax(w, h);
    sm.dc[c] = (sum + (denom >> 1)) >> vlog2(denom);
  }
  if (dm > 1 && dmp.angle < 0) {
    SlotInfo s = {};
    s.kind = 2; s.mode = dm; s.p = dmp;
#pragma unroll 1
    for (int c = 0; c < 2; c++) {
      s.set = c;
      build_projected_line(sm.proj[c], sm, s, dmp.is_ver ? w : h, dmp.is_ver ? h : w, lane, 32);
    }
  }
  __syncwarp();
  return sh;
}

// candidate `mode` (0..66 or an LM mode, DM resolved) of component comp, as chroma_predict_piece reads it.  LM modes of a visit without
// cclm get shadow parameters (nothing of theirs is stored).
__device__ __forceinline__ ChromaCand chroma_make_cand(const ChromaSmem& sm, const Rom& rom, const Shape& sh, int mode, int comp, bool cclm)
{
  ChromaCand cd;
  cd.comp = comp;
  cd.kind = mode == 0 ? 0 : mode == 1 ? 1 : mode < VVCB_LM_CHROMA ? 2 : 3;
  cd.p = rom.mode[sh.lw - 2][sh.lh - 2][mode < VVCB_LM_CHROMA ? mode : 0];
  cd.dc = sm.dc[comp];
  const int lm = vmin(vmax(mode - VVCB_LM_CHROMA, 0), 2);
  cd.a = sm.lm[lm][comp][0]; cd.k = sm.lm[lm][comp][1]; cd.b = sm.lm[lm][comp][2];
  if (cd.kind == 3 && !cclm) { cd.a = 0; cd.k = 0; cd.b = 0; }
  return cd;
}

__global__ void __launch_bounds__(kChromaWarps * 32) chroma_eval_kernel(ChromaParams P)
{
  __shared__ ChromaSmem smem[kChromaWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ChromaSmem& sm = smem[warp];
  const Rom& rom = *P.rom;
  const uint32_t* filt = &rom.filt[0][0];        // not read by the linear interpolation; a valid address for pred_angular_unit's table pointer
  const int maxv = (1 << P.bd) - 1;
  for (int vi = blockIdx.x * kChromaWarps + warp; vi < P.n; vi += gridDim.x * kChromaWarps) {
    const vvcb_chroma_visit cv = P.visits[vi];
    const Shape sh = chroma_visit_setup(sm, P, rom, cv, lane);
    const int w = sh.w, h = sh.h, dm = cv.dm_mode;

    // ---- 3. evaluations: task = (candidate * 2 + component) * lanes + unit
    const int lanes = sh.lanes, lgL = sh.lgLanes;
    int16_t* pout = P.predOut ? P.predOut + P.predOff[vi] : nullptr;
#pragma unroll 1
    for (int base = 0; base < (16 << lgL); base += 32) {
      const int task = base + lane;
      const int e = vmin(task >> lgL, 15), u = task & (lanes - 1);
      const int c = e >> 1, comp = e & 1;
      const int code = chroma_cand_code(c, dm);
      const int mode = code == VVCB_DM_CHROMA ? dm : code;
      const bool act = (task >> lgL) < 16 && (mode < VVCB_LM_CHROMA || cv.cclm);
      const ChromaCand cd = chroma_make_cand(sm, rom, sh, mode, comp, cv.cclm);
      const int16_t* org = sm.org[comp];
      int16_t* outBlk = pout ? pout + (size_t)e * w * h : nullptr;
      int sad = 0, satd = 0;
      if (sh.S == 8) {
        // an 8x8 unit as two 4x8 halves (the luma evaluation kernels' scheme): rows and the first two column stages inside a half, the
        // stage across the halves folded into the absolute sum, the 16x8 / 8x16 stage across units a butterfly with the partner lane
        const int ux = u & (sh.unitsX - 1), uy = u >> sh.lgTilesX;
        const int x0 = ux * 8, y0 = uy * 8;
        const int partnerMask = sh.tile == 4 ? 1 : sh.unitsX;
        const bool owner = sh.tile == 4 ? (ux & 1) == 0 : (uy & 1) == 0;
        uint32_t c0[4][4];
        int t = 0;
#pragma unroll 1
        for (int k = 0; k < 2; k++) {
          int q[4][8], d[4][8];
          chroma_predict_piece<4, 8>(sm, cd, sh, filt, maxv, x0, y0 + 4 * k, q);
          if (outBlk && act) store_pred<4, 8>(outBlk, w, x0, y0 + 4 * k, false, q);
          residual_unit<4, 8, false>(org + (y0 + 4 * k) * w + x0, w, q, d, sad);
          wht_rows_rc<4, 8>(d);
          wht_cols_rc<4, 8>(d);
          if (sh.tile != 3) {
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
              for (int j = 0; j < 8; j++) {
                const int other = __shfl_xor_sync(0xffffffffu, d[i][j], partnerMask);
                d[i][j] = owner ? d[i][j] + other : d[i][j] - other;
              }
          }
          if (k == 0) {
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
              for (int j = 0; j < 4; j++) c0[i][j] = pack_u16x2(vabs(d[i][2 * j]), vabs(d[i][2 * j + 1]));
          } else {
#pragma unroll
            for (int i = 0; i < 4; i++)
#pragma unroll
              for (int j = 0; j < 4; j++) t = add_halves_u16x2(max_u16x2(c0[i][j], pack_u16x2(vabs(d[i][2 * j]), vabs(d[i][2 * j + 1]))), t);
          }
        }
        if (sh.tile == 3) satd = (2 * t + 2) >> 2;                              // CL/RdCost.cpp:2306
        else {
          t += __shfl_xor_sync(0xffffffffu, t, partnerMask);
          satd = owner ? satd_norm_rect(2 * t, true) : 0;                        // CL/RdCost.cpp:2452, :2589
        }
      } else {
        // a side of 4: a lane owns one SATD tile, one (4x4) or two (8x4, 4x8) 4x4 pieces
        const int tx = u & ((1 << sh.lgTilesX) - 1), ty = u >> sh.lgTilesX;
        uint32_t c0[4][2];
        int t = 0;
#pragma unroll 1
        for (int k = 0; k < (sh.tile == 0 ? 1 : 2); k++) {
          const int x0 = tx * (sh.tile == 1 ? 8 : 4) + (sh.tile == 1 ? 4 * k : 0);
          const int y0 = ty * (sh.tile == 2 ? 8 : 4) + (sh.tile == 2 ? 4 * k : 0);
          int q[4][4], d[4][4];
          chroma_predict_piece<4, 4>(sm, cd, sh, filt, maxv, x0, y0, q);
          if (outBlk && act) store_pred<4, 4>(outBlk, w, x0, y0, false, q);
          residual_unit<4, 4, false>(org + y0 * w + x0, w, q, d, sad);
          wht_rows<4>(d);
          if (sh.tile == 0) {
            satd = (wht_cols_abs_sum<4>(d) + 1) >> 1;                            // CL/RdCost.cpp:2209
          } else {
            wht_cols<4>(d);
            if (k == 0) {
#pragma unroll
              for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 2; j++) c0[i][j] = pack_u16x2(vabs(d[i][2 * j]), vabs(d[i][2 * j + 1]));
            } else {
#pragma unroll
              for (int i = 0; i < 4; i++)
#pragma unroll
                for (int j = 0; j < 2; j++) t = add_halves_u16x2(max_u16x2(c0[i][j], pack_u16x2(vabs(d[i][2 * j]), vabs(d[i][2 * j + 1]))), t);
            }
          }
        }
        if (sh.tile != 0) satd = satd_norm_rect(2 * t, false);                  // CL/RdCost.cpp:2662, :2741
      }
      for (int o = lanes >> 1; o > 0; o >>= 1) {
        sad  += __shfl_xor_sync(0xffffffffu, sad, o);
        satd += __shfl_xor_sync(0xffffffffu, satd, o);
      }
      if (u == 0 && (task >> lgL) < 16) {
        vvcb_chroma_result& r = P.results[vi];
        r.sad[c][comp]  = act ? (uint32_t)sad : VVCB_SAT_NONE;
        r.satd[c][comp] = act ? (uint32_t)satd : VVCB_SAT_NONE;
        if (comp == 0) r.mode[c] = (uint8_t)code;
      }
    }
  }
}

// ---- chroma TU coding (vvcb_chroma_tu_eval) ----------------------------------------------------------------------------------------
// Prediction and residual of one candidate per warp, both components, into the candidate's dense blocks (Cb at the Cb TU job's offset,
// Cr behind it): the visit setup and chroma_predict_piece of chroma_eval_kernel, a lane per 4x4 piece.  Lane 0 also writes Cb's
// cbfDeltaBits (Ctx::QtCbf[Cb](0) of the candidate's snapshot) into its TU job.
struct ChromaTuPredParams {
  ChromaParams planes;                     // visits, planes, bit depth, CTU size, ROM (results / predOut are not used)
  const vvcb_chroma_tu_job* jobs; int n;
  vvcb_tu_job* cbJobs;                     // the Cb TU job of each candidate (offset read, cbf_delta_bits written)
  const vvcb_chroma_ctx_states* states;    // the candidate's snapshot (carried copy)
  int16_t* pred; int16_t* resi;
  const uint32_t* frac;                    // ProbModelTables::m_binFracBits
  const vvcb_chroma_joint_tu_job* joint;   // the joint instantiation's candidates (read instead of jobs)
};

// the forward combination of joint Cb-Cr (include/vvc_intra_b200.h): C division, truncating toward zero
__host__ __device__ __forceinline__ int chroma_joint_combine(int cb, int cr, int mode, int sign)
{
  return mode == 2 ? (cb + sign * cr) / 2 : mode == 1 ? (4 * cb + 2 * sign * cr) / 5 : (4 * cr + 2 * sign * cb) / 5;
}

__device__ __forceinline__ int32_t chroma_cbf_delta_bits(const vvcb_bin_model& m, const uint32_t* frac)
{
  const int q = ((int)m.state[0] + (int)m.state[1]) >> 8;
  return (int32_t)frac[2 * q + 1] - (int32_t)frac[2 * q];
}

// JOINT (vvcb_chroma_joint_tu_eval): both predictions at the TU job's offset as above, the combined residual of the job's mode and sign
// into the coded block, and the coded component's cbfDeltaBits (Ctx::QtCbf[Cr](0) for mode 3, else Ctx::QtCbf[Cb](0)).
template <bool JOINT = false>
__global__ void __launch_bounds__(kChromaWarps * 32) chroma_tu_pred_kernel(ChromaTuPredParams P)
{
  __shared__ ChromaSmem smem[kChromaWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  ChromaSmem& sm = smem[warp];
  const Rom& rom = *P.planes.rom;
  const uint32_t* filt = &rom.filt[0][0];
  const int maxv = (1 << P.planes.bd) - 1;
  for (int q = blockIdx.x * kChromaWarps + warp; q < P.n; q += gridDim.x * kChromaWarps) {
    uint32_t visit; uint8_t cand;
    if constexpr (JOINT) { visit = P.joint[q].visit; cand = P.joint[q].cand; }
    else { const vvcb_chroma_tu_job job = P.jobs[q]; visit = job.visit; cand = job.cand; }
    const vvcb_chroma_visit cv = P.planes.visits[visit];
    const Shape sh = chroma_visit_setup(sm, P.planes, rom, cv, lane);
    const int w = sh.w, n = sh.w * sh.h;
    const int code = chroma_cand_code(cand, cv.dm_mode), mode = code == VVCB_DM_CHROMA ? cv.dm_mode : code;
    const size_t off = P.cbJobs[q].offset;
    if constexpr (JOINT) {
      const int jm = P.joint[q].mode, sign = P.joint[q].sign;
      const ChromaCand cb = chroma_make_cand(sm, rom, sh, mode, 0, cv.cclm), cr = chroma_make_cand(sm, rom, sh, mode, 1, cv.cclm);
      int16_t* pred = P.pred + off;
      int16_t* resi = P.resi + off;
      for (int u = lane; u < (n >> 4); u += 32) {
        const int x0 = (u & ((w >> 2) - 1)) << 2, y0 = (u >> (sh.lw - 2)) << 2;
        int vb[4][4], vr[4][4];
        chroma_predict_piece<4, 4>(sm, cb, sh, filt, maxv, x0, y0, vb);
        chroma_predict_piece<4, 4>(sm, cr, sh, filt, maxv, x0, y0, vr);
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const int s = (y0 + i) * w + x0 + j;
            pred[s] = (int16_t)vb[i][j];
            pred[n + s] = (int16_t)vr[i][j];
            resi[s] = (int16_t)chroma_joint_combine(sm.org[0][s] - vb[i][j], sm.org[1][s] - vr[i][j], jm, sign);
          }
      }
      if (lane == 0) P.cbJobs[q].cbf_delta_bits = chroma_cbf_delta_bits(jm == 3 ? P.states[q].cbf_cr[0] : P.states[q].cbf_cb[0], P.frac);
    } else {
#pragma unroll 1
      for (int comp = 0; comp < 2; comp++) {
        const ChromaCand cd = chroma_make_cand(sm, rom, sh, mode, comp, cv.cclm);
        int16_t* pred = P.pred + off + (size_t)comp * n;
        int16_t* resi = P.resi + off + (size_t)comp * n;
        for (int u = lane; u < (n >> 4); u += 32) {
          const int x0 = (u & ((w >> 2) - 1)) << 2, y0 = (u >> (sh.lw - 2)) << 2;
          int v[4][4];
          chroma_predict_piece<4, 4>(sm, cd, sh, filt, maxv, x0, y0, v);
#pragma unroll
          for (int i = 0; i < 4; i++)
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const int s = (y0 + i) * w + x0 + j;
              pred[s] = (int16_t)v[i][j];
              resi[s] = (int16_t)(sm.org[comp][s] - v[i][j]);
            }
        }
      }
      if (lane == 0) P.cbJobs[q].cbf_delta_bits = chroma_cbf_delta_bits(P.states[q].cbf_cb[0], P.frac);
    }
    __syncwarp();
  }
}

// The cbf bins of xGetIntraFracBitsQT (CABACWriter::cbf_comp, context DeriveCtx::CtxQtCbf) on the candidate's carried models, one thread
// per candidate.  Step 1, after Cb's levels are final: Cb's cbf, its bin (context 0), and Cr's cbfDeltaBits from the Cr context that cbf
// selects.  Step 2, after Cr's: Cr's cbf and its bin.
struct ChromaCbfParams {
  int n, step;
  const vvcb_tu_result* res;               // the step's TU results (Cb for step 1, Cr for step 2)
  vvcb_tu_job* crJobs;                     // step 1: cbf_delta_bits of Cr written
  vvcb_chroma_ctx_states* states;          // carried models: the cbf contexts adapt
  uint8_t* cbf; uint32_t* cbfBits;         // [candidate][Cb, Cr]
  const uint32_t* frac;
};

__global__ void __launch_bounds__(128) chroma_cbf_kernel(ChromaCbfParams P)
{
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  vvcb_chroma_ctx_states& st = P.states[i];
  const unsigned cbf = P.res[i].abs_sum_level != 0;
  if (P.step == 1) {
    P.cbfBits[2 * i] = isp_code_bin(st.cbf_cb[0], P.frac, cbf);
    P.cbf[2 * i] = (uint8_t)cbf;
    P.crJobs[i].cbf_delta_bits = chroma_cbf_delta_bits(st.cbf_cr[cbf], P.frac);
  } else {
    P.cbfBits[2 * i + 1] = isp_code_bin(st.cbf_cr[P.cbf[2 * i]], P.frac, cbf);
    P.cbf[2 * i + 1] = (uint8_t)cbf;
  }
}

// Joint Cb-Cr after the TU chain (vvcb_chroma_joint_tu_eval), one warp per candidate: the inverse mapping of the job's mode and sign of the
// residual r the chain's RESI pass left in the coded block, both reconstructions (Cb over r, Cr behind it) and their SSE; then, when the
// coded residual has a level, tu_cb_coded_flag, tu_cr_coded_flag and tu_joint_cbcr_residual_flag on the candidate's carried models.
// These models are not the residual's, so pricing them after residual_coding gives the bits of the coding order.
struct ChromaJointParams {
  const vvcb_chroma_joint_tu_job* jobs; int n;
  const vvcb_chroma_visit* visits;
  const vvcb_tu_job* tuJobs;               // the candidate's TU job (offset)
  const vvcb_tu_result* res;               // the chain's results (the coded residual's levels)
  const int16_t* pred; int16_t* reco;
  const int16_t* orig[2]; int cstride, bd;
  vvcb_chroma_ctx_states* states;          // carried models
  vvcb_bin_model* joint;                   // carried Ctx::JointCbCrFlag models, 3 per candidate
  uint64_t* sse;                           // [candidate][Cb, Cr]
  uint8_t* cbf; uint32_t* bits;            // [candidate]; [candidate][cbf Cb, cbf Cr, joint flag]
  const uint32_t* frac;
};

// H.266 8.7.2 under TuCResMode, in int: CSign * -32768 does not fit int16
__host__ __device__ __forceinline__ void chroma_joint_inverse(int r, int mode, int sign, int& cb, int& cr)
{
  const int other = mode == 2 ? sign * r : (sign * r) >> 1;
  cb = mode == 3 ? other : r;
  cr = mode == 3 ? r : other;
}

__global__ void __launch_bounds__(128) chroma_joint_kernel(ChromaJointParams P)
{
  const int lane = threadIdx.x & 31;
  const int maxv = (1 << P.bd) - 1;
  for (int q = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5); q < P.n; q += (int)((gridDim.x * blockDim.x) >> 5)) {
    const vvcb_chroma_joint_tu_job j = P.jobs[q];
    const vvcb_chroma_visit v = P.visits[j.visit];
    const int w = 1 << v.log2w, n = w << v.log2h;
    const size_t off = P.tuJobs[q].offset;
    unsigned long long sse[2] = { 0, 0 };
    for (int s = lane; s < n; s += 32) {
      int res[2];
      chroma_joint_inverse(P.reco[off + s], j.mode, j.sign, res[0], res[1]);
#pragma unroll
      for (int c = 0; c < 2; c++) {
        const int rec = vmin(vmax((int)P.pred[off + c * n + s] + res[c], 0), maxv);
        P.reco[off + c * n + s] = (int16_t)rec;
        const int d = (int)P.orig[c][(size_t)(v.y + (s >> v.log2w)) * P.cstride + v.x + (s & (w - 1))] - rec;
        sse[c] += (unsigned long long)(d * d);
      }
    }
#pragma unroll
    for (int c = 0; c < 2; c++)
      for (int o = 16; o > 0; o >>= 1) sse[c] += __shfl_xor_sync(0xffffffffu, sse[c], o);
    if (lane == 0) {
      const unsigned cbf = P.res[q].abs_sum_level != 0;
      P.sse[2 * q] = sse[0]; P.sse[2 * q + 1] = sse[1];
      P.cbf[q] = (uint8_t)cbf;
      if (cbf) {
        const unsigned cbfCb = j.mode != 3, cbfCr = j.mode != 1;
        vvcb_chroma_ctx_states& st = P.states[q];
        P.bits[3 * q] = isp_code_bin(st.cbf_cb[0], P.frac, cbfCb);
        P.bits[3 * q + 1] = isp_code_bin(st.cbf_cr[cbfCb], P.frac, cbfCr);
        P.bits[3 * q + 2] = isp_code_bin(P.joint[3 * q + 2 * cbfCb + cbfCr - 1], P.frac, 1);
      }
    }
  }
}

}  // namespace
