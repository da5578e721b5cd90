// vvc_intra_b200 -- device core of the rough-mode-decision (RMD) engine.
//
// Everything here is per-lane code (no warp collectives), written as __host__ __device__ so that the
// identical source can be stepped through on a CPU by tests/host_emul.cpp (test-only lane emulation;
// the product library contains the device instantiation only and has no CPU path).
//
// Reference behaviour restated here (CL/ = VVC_project/source/Lib/CommonLib/, EL/ = .../EncoderLib/):
//   reference lines        CL/IntraPrediction.cpp:1215-1522 (xFillReferenceSamples, xFilterReferenceSamples)
//   mode parameters        CL/IntraPrediction.cpp:287-303, 487-618 (getWideAngle, initPredIntraParams)
//   planar / DC / angular  CL/IntraPrediction.cpp:248-285, 316-398, 426-479, 633-935
//   MIP                    CL/MatrixIntraPrediction.cpp:71-124, 211-254, 469-567, 637-741
//   SAD / SATD             CL/RdCost.cpp:449-484, 2118-2861
#pragma once
#include <stdint.h>
#include "../../include/vvc_intra_b200.h"

#if defined(__CUDACC__)
#define VHD __host__ __device__ __forceinline__
#else
#define VHD inline
#endif

namespace vvcb {

// ---- geometry -------------------------------------------------------------------------------------
constexpr int kLineMax   = 140;            // samples per reference line (2*64 + 1 + 3, padded)
constexpr int kNumSets   = 4;              // 0: line 0 unfiltered, 1: line 0 filtered, 2: line 1, 3: line 3
constexpr int kSlotLineWords = 54 * 32;    // int16 per warp for per-slot scratch in flight (projected main lines, MIP planes): 8x8 MIP needs 16 + 32 per lane; 54 int16 =
                                           // 27 words per lane: word aligned (projected lines are copied in words), odd word stride over the banks
constexpr int kNumClasses = 6;             // SATD tile of the shape: 0 4x4, 1 8x4, 2 4x8, 3 8x8, 4 16x8, 5 8x16
constexpr int kNumKinds   = 3;             // 0 angular, 1 planar/DC, 2 MIP
constexpr int kNumBuckets = kNumClasses * kNumKinds;
#ifndef VVCB_ITEM_TASKS
#define VVCB_ITEM_TASKS 512
#endif
constexpr int kItemTasks = VVCB_ITEM_TASKS;  // lane-tasks per plain work item (16 warp iterations; 128 -> 512: 2.4 % fewer line set-ups, profiles/r1z_summary.md)

VHD int vmin(int a, int b) { return a < b ? a : b; }
VHD int vmax(int a, int b) { return a > b ? a : b; }
VHD int vabs(int a) { return a < 0 ? -a : a; }
VHD int vlog2(int v)
{
#if defined(__CUDA_ARCH__)
  return 31 - __clz(v);
#else
  return 31 - __builtin_clz((unsigned)v);
#endif
}
// |a - b| + c (one VABSDIFF on the device)
VHD int vsad(int a, int b, int c)
{
#if defined(__CUDA_ARCH__)
  return (int)__sad(a, b, (unsigned)c);
#else
  return c + (a < b ? b - a : a - b);
#endif
}

// ---- absolute Hadamard coefficients as u16 pairs ---------------------------------------------------------------------------------
// |coefficient| of a 4x8 half stays below 2^16 (10-bit residual x 8 x 4, x 2 for the 16x8 / 8x16 partner stage), so the first half's
// values are kept two per register; the fold over the halves, sum of max(|a|, |b|), is one packed unsigned max (VIMNMX.U16x2) and
// one dot product with (1, 1) (IDP.2A.U16.U8) per pair.
VHD uint32_t pack_u16x2(int lo, int hi) { return (uint32_t)lo | ((uint32_t)hi << 16); }
VHD uint32_t max_u16x2(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
  return __vmaxu2(a, b);
#else
  const uint32_t al = a & 0xffffu, bl = b & 0xffffu, ah = a >> 16, bh = b >> 16;
  return (al > bl ? al : bl) | ((ah > bh ? ah : bh) << 16);
#endif
}
VHD int add_halves_u16x2(uint32_t w, int acc)
{
#if defined(__CUDA_ARCH__)
  return (int)__dp2a_lo(w, 0x00000101u, (unsigned)acc);
#else
  return acc + (int)(w & 0xffffu) + (int)(w >> 16);
#endif
}

// c + the signed int16 pair a times the signed int8 pair in bytes 0, 1 (lo) or 2, 3 (hi) of b: one IDP.2A.S16.S8 on the device
VHD int dot2_s16_s8_lo(uint32_t a, uint32_t b, int c)
{
#if defined(__CUDA_ARCH__)
  return __dp2a_lo((int)a, (int)b, c);
#else
  return c + (int)(int16_t)(a & 0xffffu) * (int)(int8_t)(b & 0xffu) + (int)(int16_t)(a >> 16) * (int)(int8_t)((b >> 8) & 0xffu);
#endif
}
VHD int dot2_s16_s8_hi(uint32_t a, uint32_t b, int c)
{
#if defined(__CUDA_ARCH__)
  return __dp2a_hi((int)a, (int)b, c);
#else
  return c + (int)(int16_t)(a & 0xffffu) * (int)(int8_t)((b >> 16) & 0xffu) + (int)(int16_t)(a >> 16) * (int)(int8_t)(b >> 24);
#endif
}

// Per (shape, mode) prediction parameters, precomputed on the host at context creation.
struct ModeParam {
  int16_t  angle;        // intraPredAngle (signed)
  uint16_t inv_angle;    // invAngle
  uint8_t  is_ver;
  uint8_t  ref_filter;   // use the [1 2 1]-filtered line
  uint8_t  interp;       // Gaussian 4-tap instead of the cubic one
  uint8_t  pdpc;
  int8_t   ang_scale;
  uint8_t  pad[3];
};

VHD int wide_angle(int w, int h, int mode)
{
  const int shiftTab[6] = { 0, 6, 10, 12, 14, 15 };
  if (mode > 1 && mode <= 66) {
    const int d = vabs(vlog2(w) - vlog2(h));
    if (w > h && mode < 2 + shiftTab[d]) mode += 65;
    else if (h > w && mode > 66 - shiftTab[d]) mode -= 65;
  }
  return mode;
}

// initPredIntraParams for a luma CU, no ISP / BDPCM / MIP.
VHD ModeParam make_mode_param(int w, int h, int mode, int mrl)
{
  const int angTab[32] = { 0, 1, 2, 3, 4, 6, 8, 10, 12, 14, 16, 18, 20, 23, 26, 29,
                           32, 35, 39, 45, 51, 57, 64, 73, 86, 102, 128, 171, 256, 341, 512, 1024 };
  const int invTab[32] = { 0, 16384, 8192, 5461, 4096, 2731, 2048, 1638, 1365, 1170, 1024, 910, 819, 712, 630, 565,
                           512, 468, 420, 364, 321, 287, 256, 224, 191, 161, 128, 96, 64, 48, 32, 16 };
  const int filtThr[8] = { 24, 24, 24, 14, 2, 0, 0, 0 };
  ModeParam p = {};
  const int predMode = wide_angle(w, h, mode);
  p.is_ver = predMode >= 34;
  p.pdpc   = mrl == 0;           // w,h >= 4 always holds for luma CUs
  int absAng = 0;
  const int angMode = p.is_ver ? predMode - 50 : -(predMode - 18);
  if (mode > 1) {
    const int a = vabs(angMode);
    absAng      = angTab[a];
    p.inv_angle = (uint16_t)invTab[a];
    p.angle     = (int16_t)(angMode < 0 ? -absAng : absAng);
    if (angMode < 0) p.pdpc = 0;
    else if (angMode > 0) {
      const int side = p.is_ver ? h : w;
      const int sc   = vmin(2, vlog2(side) - (vlog2(3 * p.inv_angle - 2) - 8));
      p.ang_scale = (int8_t)sc;
      p.pdpc = p.pdpc && sc >= 0;
    }
  }
  if (mrl || mode == 1) return p;
  if (mode == 0) { p.ref_filter = w * h > 32; return p; }
  const int diff = vmin(vabs(predMode - 18), vabs(predMode - 50));
  if (diff > filtThr[(vlog2(w) + vlog2(h)) >> 1]) {
    const bool integerSlope = (absAng & 31) == 0;
    p.ref_filter = integerSlope;
    p.interp     = !integerSlope;
  }
  return p;
}

// initPredIntraParams for a prediction region (pw x ph) of an intra sub-partition CU (cuW x cuH): the wide-angle remap takes the CU's
// shape, PDPC and its scale the region's; no reference smoothing, cubic interpolation only, reference line 0 (CL/IntraPrediction.cpp:
// 492-511, :544-551, :558-574 with JVET_O0502_ISP_CLEANUP).  Host side of vvcb_isp_mode_param.
VHD ModeParam make_mode_param_isp(int cuW, int cuH, int pw, int ph, int mode)
{
  ModeParam p = make_mode_param(cuW, cuH, mode, 1);      // reference line 1: angle fields only, no filters, no PDPC
  p.pdpc = pw >= 4 && ph >= 4;
  p.ang_scale = 0;
  if (mode > 1 && p.angle < 0) p.pdpc = 0;
  else if (mode > 1 && p.angle > 0) {
    const int sc = vmin(2, vlog2(p.is_ver ? ph : pw) - (vlog2(3 * p.inv_angle - 2) - 8));
    p.ang_scale = (int8_t)sc;
    p.pdpc = p.pdpc && sc >= 0;
  }
  return p;
}

VHD int mip_num_modes(int w, int h)
{
  if (w > 4 * h || h > 4 * w) return 0;
  if (w == 4 && h == 4) return 35;
  if (w <= 8 && h <= 8) return 19;
  return 11;
}

// ---- work decomposition ---------------------------------------------------------------------------
// A visit is cut into square "units" of S x S samples (S = 4 when min(w,h) == 4, else 8); one lane
// predicts one unit (two for the 8x4 / 4x8 SATD tiles) and keeps its residual in registers.
struct Shape {
  int w, h, lw, lh;
  int S;              // unit size
  int unitsX, unitsY; // units per row / column of the CU
  int lanes;          // lanes per evaluation slot (power of two, 1..64)
  int tile;           // SATD tile: 0 4x4, 1 8x4, 2 4x8, 3 8x8, 4 16x8, 5 8x16
  int lgLanes;        // log2(lanes)
  int lgTilesX;       // log2 of the lane grid width: units per row (S == 8) or SATD tiles per row (S == 4)
};

VHD Shape make_shape(int lw, int lh)
{
  Shape s;
  s.lw = lw; s.lh = lh; s.w = 1 << lw; s.h = 1 << lh;
  const int w = s.w, h = s.h;
  if      (w > h && (h & 7) == 0 && (w & 15) == 0) s.tile = 4;
  else if (w < h && (w & 7) == 0 && (h & 15) == 0) s.tile = 5;
  else if (w > h && (w & 7) == 0)                  s.tile = 1;
  else if (w < h && (h & 7) == 0)                  s.tile = 2;
  else if ((w & 7) == 0 && (h & 7) == 0)           s.tile = 3;
  else                                             s.tile = 0;
  s.S = (w == 4 || h == 4) ? 4 : 8;
  s.unitsX = w / s.S; s.unitsY = h / s.S;
  // 8x4 / 4x8 tiles: one lane owns both 4x4 units of a tile
  s.lanes = (s.tile == 1 || s.tile == 2) ? (w * h) / 32 : s.unitsX * s.unitsY;
  s.lgLanes  = vlog2(s.lanes);
  s.lgTilesX = s.S == 8 ? lw - 3 : (s.tile == 1 ? lw - 3 : lw - 2);
  return s;
}

struct WorkItem {            // 8 bytes
  uint32_t visit;
  uint16_t slot_begin;       // index into the visit's list of active slots
  uint16_t slot_count;
};

// ---- reference lines ------------------------------------------------------------------------------
// Availability is a set of at most five intervals on the walk bottom-left -> corner -> top-right; an
// unavailable sample takes the nearest earlier available sample on the walk, or the first available one.
// UNIT: samples per availability count, 4 for luma, 2 for 4:2:0 chroma (pcv.minCUWidth >> scaleX).
struct LineGeom {
  int w, h, mrl, n;          // n = walk length
  int lo[5], hi[5];          // available intervals [lo, hi) in walk order: below-left, left, corner, above, above-right; an absent
                             // one has lo = kNoInterval (never reached).  Fixed slots, statically indexed: the struct stays in registers.
  int first;                 // first available walk position, -1 when nothing is available
};
constexpr int kNoInterval = 0x3fffffff;

template <int UNIT = 4> VHD LineGeom make_line_geom(const vvcb_rmd_visit& v, int w, int h, int mrl)
{
  LineGeom g;
  g.w = w; g.h = h; g.mrl = mrl;
  const int C = 2 * h + 2 * mrl + 1;
  g.n = C + 2 * w;
  g.lo[0] = v.n_below_left  ? h - UNIT * v.n_below_left : kNoInterval;  g.hi[0] = h;
  g.lo[1] = v.n_left        ? 2 * h - UNIT * v.n_left   : kNoInterval;  g.hi[1] = 2 * h;
  g.lo[2] = v.avail_al      ? 2 * h                     : kNoInterval;  g.hi[2] = C;
  g.lo[3] = v.n_above       ? C                         : kNoInterval;  g.hi[3] = C + UNIT * v.n_above;
  g.lo[4] = v.n_above_right ? C + w                     : kNoInterval;  g.hi[4] = C + w + UNIT * v.n_above_right;
  g.first = -1;
#pragma unroll
  for (int k = 4; k >= 0; k--) if (g.lo[k] != kNoInterval) g.first = g.lo[k];
  return g;
}

// walk position the sample at walk position i is copied from (-1: nothing available -> mid-grey)
VHD int line_source(const LineGeom& g, int i)
{
  int src = g.first;                       // before the first interval: its first sample
#pragma unroll
  for (int k = 0; k < 5; k++)
    if (i >= g.lo[k]) src = i < g.hi[k] ? i : g.hi[k] - 1;
  return src;
}

// walk position -> (is_left, index into left[] / top[]) and picture offset relative to the CU origin
VHD void line_pos(const LineGeom& g, int i, bool& isLeft, int& k, int& dx, int& dy)
{
  const int nLeft = 2 * g.h + g.mrl;       // walk positions [0, nLeft) are left[nLeft - i]
  if (i < nLeft) { isLeft = true;  k = nLeft - i;  dx = -1 - g.mrl; dy = -1 - g.mrl + k; }
  else           { isLeft = false; k = i - nLeft;  dx = -1 - g.mrl + k; dy = -1 - g.mrl; }
}

// ---- MIP matrices for IDP.2A ---------------------------------------------------------------------------
// Per matrix family (0: 4x4, 18 modes of 16 rows x 4 weights; 1: 8x8, 10 modes of 16 x 8; 2: 16x16, 6 modes of 64 x 7) and mode: its rows
// as packed int8 weights, one word (family 0) or two words (1, 2) per row, then one header row whose first word is shift | offset << 8.
// The 16x16 family's 7 columns get a zero weight in front, standing for its first input, which that family drops (and which the input
// vector holds as 0), so a row is the dot product of the 4 or 8 inputs with two or four IDP.2A.  The header row also staggers the modes
// over the shared-memory banks (mode stride = odd number of rows): the lanes of a warp iteration reading the same row of different modes
// hit different banks.  The weights are 0..123, so they read the same as signed bytes.
VHD int mip_mode_words(int family) { return family == 0 ? 17 : (family == 1 ? 34 : 130); }
VHD int mip_family_words(int family) { return family == 0 ? 18 * 17 : (family == 1 ? 10 * 34 : 6 * 130); }
VHD int mip_family_base(int family) { return family == 0 ? 0 : (family == 1 ? 18 * 17 : 18 * 17 + 10 * 34); }
constexpr int kMipRomWords = 18 * 17 + 10 * 34 + 6 * 130;   // 5 704 bytes

// ---- 4-tap filter tables (packed int8 x4, one word per fractional position) -------------------------
struct Rom {
  uint32_t filt[2][32];                    // [0] cubic (CL/InterpolationFilter.cpp:100), [1] Gaussian (CL/IntraPrediction.cpp:76)
  ModeParam mode[6][6][VVCB_NUM_LUMA_MODE];  // [log2w-2][log2h-2][mode], reference line 0
  uint8_t angOrder[6][6][65];              // angular modes 2..66 ordered by (hor/ver, PDPC class) so that the lanes of a warp agree
  alignas(16) uint32_t mip[kMipRomWords];  // MIP matrices, shifts and offsets in the layout above (two-word rows read as one 8-byte load)
};

// ---- register-resident Walsh-Hadamard pieces -------------------------------------------------------
// C-point transform of each of the R rows
template <int R, int C> VHD void wht_rows_rc(int (&d)[R][C])
{
#pragma unroll
  for (int y = 0; y < R; y++)
#pragma unroll
    for (int len = 1; len < C; len <<= 1)
#pragma unroll
      for (int i = 0; i < C; i += 2 * len)
#pragma unroll
        for (int x = i; x < i + len; x++) {
          const int a = d[y][x], b = d[y][x + len];
          d[y][x] = a + b; d[y][x + len] = a - b;
        }
}
template <int N> VHD void wht_rows(int (&d)[N][N]) { wht_rows_rc<N, N>(d); }

// R-point transform of each of the C columns (all stages)
template <int R, int C> VHD void wht_cols_rc(int (&d)[R][C])
{
#pragma unroll
  for (int x = 0; x < C; x++)
#pragma unroll
    for (int len = 1; len < R; len <<= 1)
#pragma unroll
      for (int i = 0; i < R; i += 2 * len)
#pragma unroll
        for (int y = i; y < i + len; y++) {
          const int a = d[y][x], b = d[y + len][x];
          d[y][x] = a + b; d[y + len][x] = a - b;
        }
}

// columns, all stages but the last; the last stage is folded into the absolute sum:
// |a+b| + |a-b| = 2 max(|a|, |b|)
template <int N> VHD int wht_cols_abs_sum(int (&d)[N][N])
{
#pragma unroll
  for (int x = 0; x < N; x++)
#pragma unroll
    for (int len = 1; len < N / 2; len <<= 1)
#pragma unroll
      for (int i = 0; i < N; i += 2 * len)
#pragma unroll
        for (int y = i; y < i + len; y++) {
          const int a = d[y][x], b = d[y + len][x];
          d[y][x] = a + b; d[y + len][x] = a - b;
        }
  int s = 0;
#pragma unroll
  for (int x = 0; x < N; x++)
#pragma unroll
    for (int y = 0; y < N / 2; y++) s += vmax(vabs(d[y][x]), vabs(d[y + N / 2][x]));
  return 2 * s;
}

template <int N> VHD void wht_cols(int (&d)[N][N]) { wht_cols_rc<N, N>(d); }

// (int)(s / sqrt(N) * 2) of CL/RdCost.cpp:2452,2589,2662,2741 as one multiply; exactness over the
// reachable range of s is proven exhaustively in tests/test_oracle_golden.py.
VHD int satd_norm_rect(int s, bool is128)
{
  const double c = is128 ? 0.17677669529663687 /* 2/sqrt(128) */ : 0.35355339059327373 /* 2/sqrt(32) */;
  return (int)((double)s * c);
}

// ---- prediction of one S x S unit ------------------------------------------------------------------
struct SlotInfo {
  int  kind;            // 0 planar, 1 DC, 2 angular, 3 MIP
  int  mode, mrl, set;  // set: which reference-line set feeds the prediction
  ModeParam p;
};

// clip to [0, maxv]: one VIMNMX.RELU on the device
VHD int clip_bd(int v, int maxv)
{
#if defined(__CUDA_ARCH__)
  return __vimin_s32_relu(v, maxv);
#else
  return vmin(vmax(v, 0), maxv);
#endif
}

// Angular prediction of the unit whose origin is (c0, r0) in the main/side frame.  ml points at the
// slot's main line so that ml[t] == refMain0[t] (may be indexed with negative t); side points at
// refSide0.  Output in the main/side frame: q[r][c].  LINEAR: the 2-tap linear interpolation of chroma blocks
// ((32 - f) * refMain[x + dInt + 1] + f * refMain[x + dInt + 2] + 16) >> 5 instead of the 4-tap luma filters (filt must still point at the table; its taps are unused).
template <int R, int C, bool LINEAR = false> VHD void pred_angular_unit(const int16_t* ml, const int16_t* side, const ModeParam& p, int mrl,
                                                   int mw, int mh, int c0, int r0, const uint32_t* filt, int maxv, int (&q)[R][C])
{
  const int angle = p.angle;
  const uint32_t* ftab = filt + (p.interp ? 32 : 0);
#pragma unroll
  for (int i = 0; i < R; i++) {
    const int r   = r0 + i;
    const int pos = angle * (r + 1 + mrl);
    const int dInt = pos >> 5, dFrac = pos & 31;
    const uint32_t fw = ftab[dFrac];
    const int f0 = (int)(int8_t)(fw & 0xff), f1 = (int)(int8_t)((fw >> 8) & 0xff);
    const int f2 = (int)(int8_t)((fw >> 16) & 0xff), f3 = (int)(int8_t)(fw >> 24);
    const int16_t* m = ml + mrl + dInt + c0;
    int t[C + 3];
#pragma unroll
    for (int j = 0; j < C + 3; j++) t[j] = m[j];
#pragma unroll
    for (int j = 0; j < C; j++) {
      if constexpr (LINEAR) q[i][j] = ((32 - dFrac) * t[j + 1] + dFrac * t[j + 2] + 16) >> 5;
      else q[i][j] = clip_bd((f0 * t[j] + f1 * t[j + 1] + f2 * t[j + 2] + f3 * t[j + 3] + 32) >> 6, maxv);
    }
  }
  #ifdef VVCB_EXP_NO_PDPC
  if (false) {
#else
  if (p.pdpc) {
#endif
    if (angle == 0) {
      const int scale = (vlog2(mw) + vlog2(mh) - 2) >> 2;
      const int lim = vmin(3 << scale, mw);
      const int tl = ml[0];
#pragma unroll
      for (int j = 0; j < C; j++) {
        const int c = c0 + j;
        if (c < lim) {
          const int wL = 32 >> ((2 * c) >> scale);
#pragma unroll
          for (int i = 0; i < R; i++)
            q[i][j] = clip_bd(q[i][j] + ((wL * (side[1 + r0 + i] - tl) + 32) >> 6), maxv);
        }
      }
    } else {
      const int scale = p.ang_scale;
      const int lim = vmin(3 << scale, mw);
#pragma unroll
      for (int j = 0; j < C; j++) {
        const int c = c0 + j;
        if (c < lim) {
          const int wL  = 32 >> ((2 * c) >> scale);
          const int off = (256 + (c + 1) * (int)p.inv_angle) >> 9;
#pragma unroll
          for (int i = 0; i < R; i++) {
            const int l = side[r0 + i + off + 1];
            q[i][j] = q[i][j] + ((wL * (l - q[i][j]) + 32) >> 6);
          }
        }
      }
    }
  }
}

// Planar / DC (+PDPC) of the unit at block position (x0, y0); output in block orientation b[y][x].
template <int R, int C> VHD void pred_planar_dc_unit(const int16_t* top, const int16_t* left, int kind, bool pdpc, int dc,
                                                     int lw, int lh, int x0, int y0, int (&b)[R][C])
{
  const int w = 1 << lw, h = 1 << lh;
  const int tr = top[w + 1], bl = left[h + 1];
  const int scale = (lw + lh - 2) >> 2;
#pragma unroll
  for (int i = 0; i < R; i++) {
    const int y = y0 + i;
    const int l = left[y + 1];
    const int wT = 32 >> vmin(31, (y << 1) >> scale);
#pragma unroll
    for (int j = 0; j < C; j++) {
      const int x = x0 + j;
      const int t = top[x + 1];
      int v;
      if (kind == 0) {
        const int hor = (l << lw) + (x + 1) * (tr - l);
        const int ver = (t << lh) + (y + 1) * (bl - t);
        v = ((hor << lh) + (ver << lw) + (1 << (lw + lh))) >> (1 + lw + lh);
      } else v = dc;
      if (pdpc) {
        const int wL = 32 >> vmin(31, (x << 1) >> scale);
        v = v + ((wL * (l - v) + wT * (t - v) + 32) >> 6);
      }
      b[i][j] = v;
    }
  }
}

// ---- MIP --------------------------------------------------------------------------------------------
struct MipGeom {
  int numModes, small, bsz, redW, redH, upH, upV, grid;
  int lgRedW, lgUpH, lgUpV;
  int family;            // 0: 4x4 matrices (4 inputs), 1: 8x8 matrices (8 inputs), 2: 16x16 matrices (7 inputs, first column dropped)
};

VHD MipGeom make_mip_geom(int w, int h)
{
  MipGeom g;
  g.numModes = mip_num_modes(w, h);
  g.small = w <= 8 && h <= 8;
  g.bsz   = (w > 4 || h > 4) ? 4 : 2;
  g.redW  = g.small ? 4 : vmin(w, 8);
  g.redH  = g.small ? 4 : vmin(h, 8);
  g.upH   = w / g.redW; g.upV = h / g.redH;
  g.grid  = g.small ? 4 : 8;
  g.lgRedW = vlog2(g.redW); g.lgUpH = vlog2(g.upH); g.lgUpV = vlog2(g.upV);
  g.family = (w == 4 && h == 4) ? 0 : (g.small ? 1 : 2);
  return g;
}

// Everything one MIP mode needs besides the visit's boundary (CL/MatrixIntraPrediction.cpp:211-254, 570-591)
struct MipSlot {
  const uint32_t* mat;   // the mode's rows in Rom::mip's layout
  int shift, off, inOff;
  bool transpose;
  uint32_t in[4];        // rebased reduced boundary (zero padded) as int16 pairs; input 0 is 0 for the 16x16 family
};

// famRom: g.family's part of Rom::mip (in global memory or a shared-memory copy); mipIn[t][i]: rebased input vector of orientation t
// (0 normal, 1 transposed), word aligned; mipAux: {inOff[0], inOff[1], sum[0], sum[1]}
VHD MipSlot make_mip_slot(const uint32_t* famRom, const MipGeom& g, const int16_t (*mipIn)[8], const int* mipAux, int mode)
{
  MipSlot m;
  m.transpose = mode > g.numModes / 2;
  const int widx = m.transpose ? mode - g.numModes / 2 : mode;
  m.mat = famRom + widx * mip_mode_words(g.family);
  const uint32_t head = m.mat[g.family == 2 ? 128 : (g.family == 1 ? 32 : 16)];
  m.shift = (int)(head & 0xffu);
  const int t = m.transpose ? 1 : 0;
  const uint32_t* in2 = reinterpret_cast<const uint32_t*>(mipIn[t]);
#pragma unroll
  for (int i = 0; i < 4; i++) m.in[i] = in2[i];
  m.inOff = mipAux[t];
  m.off = (1 << (m.shift - 1)) - (int)(head >> 8) * mipAux[2 + t];
  return m;
}

// Reduced sample of matrix row `row`: WIDE = 8 inputs (8x8 and 16x16 families), else 4 (4x4 family)
template <bool WIDE> VHD int mip_row_sample(const MipSlot& m, int row, int maxv)
{
  int acc;
  if (WIDE) {
    const uint2 w = reinterpret_cast<const uint2*>(m.mat)[row];
    acc = dot2_s16_s8_lo(m.in[0], w.x, m.off);
    acc = dot2_s16_s8_hi(m.in[1], w.x, acc);
    acc = dot2_s16_s8_lo(m.in[2], w.y, acc);
    acc = dot2_s16_s8_hi(m.in[3], w.y, acc);
  } else {
    const uint32_t w = m.mat[row];
    acc = dot2_s16_s8_lo(m.in[0], w, m.off);
    acc = dot2_s16_s8_hi(m.in[1], w, acc);
  }
  return clip_bd((acc >> m.shift) + m.inOff, maxv);
}

// One sample of the reduced prediction at logical position (rx, ry), CL/MatrixIntraPrediction.cpp:637-741.
VHD int mip_reduced_sample(const MipSlot& m, const MipGeom& g, int w, int h, int maxv, int rx, int ry)
{
  bool lho = (w == 4 && h >= 16), lvo = (h == 4 && w >= 16);
  int xx = rx, yy = ry, iw = g.redW;
  if (m.transpose) { const bool t = lho; lho = lvo; lvo = t; xx = ry; yy = rx; iw = g.redH; }
  const int row = (lvo ? 2 * yy : yy) * (g.small ? iw : g.grid) + (lho ? 2 * xx : xx);
  return g.family == 0 ? mip_row_sample<false>(m, row, maxv) : mip_row_sample<true>(m, row, maxv);
}

// ---- mode bits (lists kernel) -----------------------------------------------------------------------
VHD int trunc_bin_len(int symbol, int numSymbols)
{
  const int thresh = vlog2(numSymbols);
  const int b = numSymbols - (1 << thresh);
  return symbol < (1 << thresh) - b ? thresh : thresh + 1;
}

// bits of CABACWriter::intra_luma_pred_mode on the estimator (EL/CABACWriter.cpp:1762-1845)
VHD uint64_t mode_bits(const vvcb_rates& r, const uint8_t* mpm, int w, int h, bool mrlAllowed, bool mipEnabled,
                       bool isMip, int mrl, int mode)
{
  const uint64_t EP = 1u << 15;
  uint64_t bits = 0;
  const int numMip = mip_num_modes(w, h);
  if (mipEnabled && numMip) bits += r.mip_flag[isMip ? 1 : 0];
  if (isMip) return bits + EP * (uint64_t)trunc_bin_len(mode, numMip);
  if (mrlAllowed) {
    bits += r.mrl_bin0[mrl != 0];
    if (mrl != 0) bits += r.mrl_bin1[mrl != 1];
  }
  if (mrl == 0 && vlog2(w) + vlog2(h) > 4) bits += r.isp_bin0_0;
  int idx = 6;
  for (int i = 5; i >= 0; i--) if (mpm[i] == mode) idx = i;
  if (mrl == 0) bits += r.mpm_flag[idx < 6];
  if (idx < 6) {
    if (mrl == 0) bits += r.planar_flag[idx > 0];
    if (idx > 0) bits += EP * (uint64_t)vmin(idx, 4);
  } else {
    int rem = mode;
    // mode minus the number of MPMs below it == the reference's sorted descending decrement loop
    int below = 0;
    for (int i = 0; i < 6; i++) below += mpm[i] < mode;
    rem -= below;
    bits += EP * (uint64_t)trunc_bin_len(rem, 61);
  }
  return bits;
}

}  // namespace vvcb
