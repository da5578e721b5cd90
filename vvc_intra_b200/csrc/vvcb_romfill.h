// Host-side construction of the device ROM (filter words, per-shape mode parameters, MIP matrices in IDP.2A form).
#pragma once
#include <stdlib.h>
#include <string.h>
#include "vvcb_core.cuh"
#include "vvc_rom_tables.h"

namespace vvcb {
inline void fill_rom(Rom& r)
{
  memset(&r, 0, sizeof(r));
  for (int t = 0; t < 2; t++)
    for (int f = 0; f < 32; f++) {
      const int8_t* c = (t ? kIntraGaussFilter : kIntraCubicFilter) + 4 * f;
      r.filt[t][f] = (uint32_t)(uint8_t)c[0] | ((uint32_t)(uint8_t)c[1] << 8) | ((uint32_t)(uint8_t)c[2] << 16) | ((uint32_t)(uint8_t)c[3] << 24);
    }
  for (int lw = 2; lw <= 6; lw++)
    for (int lh = 2; lh <= 6; lh++)
      for (int m = 0; m < VVCB_NUM_LUMA_MODE; m++) r.mode[lw - 2][lh - 2][m] = make_mode_param(1 << lw, 1 << lh, m, 0);
  for (int lw = 2; lw <= 6; lw++)
    for (int lh = 2; lh <= 6; lh++) {
      int n = 0;
      for (int key = 0; key < 6; key++)          // key = is_ver * 3 + PDPC class (0 none, 1 angular, 2 pure hor/ver)
        for (int m = 2; m < VVCB_NUM_LUMA_MODE; m++) {
          const ModeParam& p = r.mode[lw - 2][lh - 2][m];
          const int cls = !p.pdpc ? 0 : (p.angle == 0 ? 2 : 1);
          if (p.is_ver * 3 + cls == key) r.angOrder[lw - 2][lh - 2][n++] = (uint8_t)m;
        }
    }
  // MIP matrices in Rom::mip's layout: rows of 4 or 8 int8 weights (the 16x16 family's 7 behind a zero), then the header row
  static const uint8_t* const mat[3] = { kMipMatrix4x4, kMipMatrix8x8, kMipMatrix16x16 };
  static const uint8_t* const off[3] = { kMipOffset4x4, kMipOffset8x8, kMipOffset16x16 };
  static const uint8_t* const sh[3] = { kMipShift4x4, kMipShift8x8, kMipShift16x16 };
  static const int modes[3] = { 18, 10, 6 }, rows[3] = { 16, 16, 64 }, cols[3] = { 4, 8, 7 };
  for (int f = 0; f < 3; f++)
    for (int m = 0; m < modes[f]; m++) {
      uint32_t* dst = r.mip + mip_family_base(f) + m * mip_mode_words(f);
      const int rowWords = f ? 2 : 1;
      for (int y = 0; y < rows[f]; y++)
        for (int c = 0; c < cols[f]; c++) {
          const uint8_t wgt = mat[f][(m * rows[f] + y) * cols[f] + c];
          if (wgt > 127) abort();                    // read as a signed byte by IDP.2A
          const int k = c + (f == 2 ? 1 : 0);
          dst[y * rowWords + (k >> 2)] |= (uint32_t)wgt << (8 * (k & 3));
        }
      dst[rows[f] * rowWords] = (uint32_t)sh[f][m] | ((uint32_t)off[f][m] << 8);
    }
}

}  // namespace vvcb

// forward transform kernels and quantiser scales (vvcb_tu.cuh's TrRom); T has the TrRom layout
template <class T> inline void fill_tr_rom(T& r)
{
  memset(&r, 0, sizeof(r));
  memcpy(r.dct2, kDct2_4, 32); memcpy(r.dct2 + 16, kDct2_8, 128); memcpy(r.dct2 + 80, kDct2_16, 512);
  memcpy(r.dct2 + 336, kDct2_32, 2048); memcpy(r.dct2 + 1360, kDct2_64, 8192);
  memcpy(r.dct8, kDct8_4, 32); memcpy(r.dct8 + 16, kDct8_8, 128); memcpy(r.dct8 + 80, kDct8_16, 512); memcpy(r.dct8 + 336, kDct8_32, 2048);
  memcpy(r.dst7, kDst7_4, 32); memcpy(r.dst7 + 16, kDst7_8, 128); memcpy(r.dst7 + 80, kDst7_16, 512); memcpy(r.dst7 + 336, kDst7_32, 2048);
  for (int i = 0; i < 12; i++) { r.quantScales[i] = kQuantScales[i]; r.invQuantScales[i] = kInvQuantScales[i]; }
  memcpy(r.lfnst8, kLfnst8x8, sizeof(kLfnst8x8)); memcpy(r.lfnst4, kLfnst4x4, sizeof(kLfnst4x4)); memcpy(r.lfnstLut, kLfnstLut, 95);
  int n = 0;                                           // up-right diagonal order of a 4x4 group
  for (int d = 0; d <= 6; d++) for (int y = d < 3 ? d : 3; y >= 0 && d - y <= 3; y--) r.diag4[n++] = (uint8_t)((d - y) | (y << 2));
}

// Tables of the dependent-quantisation kernel (vvcb_dq.cuh's DqRom; T has that layout): the grouped 4x4 up-right diagonal
// scan of every luma TU shape (H.266 6.5.2; CL/Rom.cpp:263-365), the template neighbourhoods inside and outside the
// sub-block (CL/DepQuant.cpp:153-303) and the Golomb-Rice tables (CL/DepQuant.cpp:887, CL/Rom.cpp:628-638).
template <class T> inline void fill_dq_rom(T& r)
{
  memset(&r, 0, sizeof(r));
  static const int32_t riceBits[4][32] = {
    { 32768,  65536,  98304, 131072, 163840, 196608, 262144, 262144, 327680, 327680, 327680, 327680, 393216, 393216, 393216, 393216, 393216, 393216, 393216, 393216, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752, 458752},
    { 65536,  65536,  98304,  98304, 131072, 131072, 163840, 163840, 196608, 196608, 229376, 229376, 294912, 294912, 294912, 294912, 360448, 360448, 360448, 360448, 360448, 360448, 360448, 360448, 425984, 425984, 425984, 425984, 425984, 425984, 425984, 425984},
    { 98304,  98304,  98304,  98304, 131072, 131072, 131072, 131072, 163840, 163840, 163840, 163840, 196608, 196608, 196608, 196608, 229376, 229376, 229376, 229376, 262144, 262144, 262144, 262144, 327680, 327680, 327680, 327680, 327680, 327680, 327680, 327680},
    {131072, 131072, 131072, 131072, 131072, 131072, 131072, 131072, 163840, 163840, 163840, 163840, 163840, 163840, 163840, 163840, 196608, 196608, 196608, 196608, 196608, 196608, 196608, 196608, 229376, 229376, 229376, 229376, 229376, 229376, 229376, 229376} };
  static const uint8_t ricePars[32] = { 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 2, 3, 3, 3, 3 };
  static const uint8_t riceZero[3][32] = {
    {0, 0, 0, 0, 0, 1, 2, 2, 2, 2, 2, 2, 4, 4, 4, 4, 4, 4,  4,  4,  4,  4,  4,  8,  8,  8,  8,  8,  8,  8,  8,  8},
    {1, 1, 1, 1, 2, 3, 4, 4, 4, 6, 6, 6, 8, 8, 8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 12, 16, 16, 16, 16, 16, 16},
    {1, 1, 2, 2, 2, 3, 4, 4, 4, 6, 6, 6, 8, 8, 8, 8, 8, 8, 12, 12, 12, 12, 12, 12, 12, 16, 16, 16, 16, 16, 16, 16} };
  static const uint8_t groupIdx[32] = { 0,1,2,3,4,4,5,5,6,6,6,6,7,7,7,7,8,8,8,8,8,8,8,8,9,9,9,9,9,9,9,9 };
  memcpy(r.goRiceBits, riceBits, sizeof(riceBits)); memcpy(r.goRicePars, ricePars, 32); memcpy(r.goRiceZero, riceZero, 96);
  memcpy(r.groupIdx, groupIdx, 32);
  static const uint8_t tsRice[32] = { 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2, 2, 2 };
  memcpy(r.tsRicePars, tsRice, 32);
  for (int i = 0; i < 12; i++) { r.quantScales[i] = kQuantScales[i]; r.invQuantScales[i] = kInvQuantScales[i]; }

  // up-right diagonal order of a bw x bh grid
  auto diag = [](int bw, int bh, int* ox, int* oy) {
    int n = 0;
    for (int d = 0; d <= bw + bh - 2; d++)
      for (int y = (d < bh - 1 ? d : bh - 1); y >= 0 && d - y < bw; y--) { ox[n] = d - y; oy[n] = y; n++; }
    return n;
  };
  int ix[16], iy[16], inId[4][4];
  diag(4, 4, ix, iy);
  for (int i = 0; i < 16; i++) inId[iy[i]][ix[i]] = i;
  // template neighbours (x+1, x+2, (x+1,y+1), y+1, y+2) that fall inside the same 4x4 sub-block, ascending scan position
  static const int dx[5] = { 1, 2, 1, 0, 0 }, dy[5] = { 0, 0, 1, 1, 2 };
  for (int i = 0; i < 16; i++) {
    int list[5], n = 0;
    for (int k = 0; k < 5; k++) { const int x = ix[i] + dx[k], y = iy[i] + dy[k]; if (x < 4 && y < 4) list[n++] = inId[y][x]; }
    for (int a = 1; a < n; a++) for (int b = a; b > 0 && list[b] < list[b - 1]; b--) { const int t = list[b]; list[b] = list[b - 1]; list[b - 1] = t; }
    r.nbIn[i][0] = (uint8_t)n;
    for (int k = 0; k < n; k++) r.nbIn[i][1 + k] = (uint8_t)list[k];
  }
  int first = 0;
  static int idOf[32][32];
  for (int lw = 2; lw <= 6; lw++)
    for (int lh = 2; lh <= 6; lh++) {
      const int w = 1 << lw, nzW = w < 32 ? w : 32, nzH = (1 << lh) < 32 ? (1 << lh) : 32;
      const int gw = nzW >> 2, gh = nzH >> 2;
      int gx[64], gy[64];
      diag(gw, gh, gx, gy);
      auto& sh = r.shape[lw - 2][lh - 2];
      sh.first = first; sh.numCoeff = nzW * nzH; sh.numSbb = gw * gh; sh.widthInSbb = gw; sh.heightInSbb = gh;
      for (int g = 0; g < gw * gh; g++) {
        r.sbbPos[lw - 2][lh - 2][g] = (uint16_t)(gy[g] * gw + gx[g]);
        for (int i = 0; i < 16; i++) {
          auto& p = r.pos[first + g * 16 + i];
          p.x = (uint8_t)(gx[g] * 4 + ix[i]); p.y = (uint8_t)(gy[g] * 4 + iy[i]); p.idx = (uint16_t)(p.y * w + p.x);
          idOf[p.y][p.x] = g * 16 + i;
        }
      }
      int runMax = 0;
      for (int id = 0; id < sh.numCoeff; id++) {
        auto& p = r.pos[first + id];
        const int beg = id & ~15;
        int list[5], n = 0;
        for (int k = 0; k < 5; k++) {
          const int x = p.x + dx[k], y = p.y + dy[k];
          if (x < nzW && y < nzH && idOf[y][x] >= beg + 16) list[n++] = idOf[y][x];
        }
        for (int a = 1; a < n; a++) for (int b = a; b > 0 && list[b] < list[b - 1]; b--) { const int t = list[b]; list[b] = list[b - 1]; list[b - 1] = t; }
        p.numOut = (uint8_t)n;
        for (int k = 0; k < n; k++) { if (list[k] > runMax) runMax = list[k]; p.outPos[k] = (uint16_t)(list[k] - beg); }
        p.maxDist = (uint16_t)(runMax > id ? runMax - id : 0);    // running maximum of the absolute positions, made relative
      }
      first += sh.numCoeff;
    }
}
