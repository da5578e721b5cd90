// vvc_intra_b200 -- TU coding kernel (sm_100a): forward separable transform (DCT-II / DST-VII / DCT-VIII as exact
// integer matrix products, or transform skip), pre-selection sum, scalar quantisation, dequantisation, inverse
// transform with the reference's intermediate clipping, reconstruction and SSE.
//
// Reference behaviour: CL/TrQuant.cpp:835-915 (xT), :917-993 (xIT), :1394-1438 / :996-1041 (transform skip),
// :1090-1103 (pre-selection sum), CL/Quant.cpp:994-1089 (quant), :423-540 (dequant), CL/RdCost.cpp:1739 (SSE).
// The reference's partial butterflies (CL/TrQuant_EMT.cpp) are exact evaluations of the same products.
// One CTA per job; the block lives in shared memory as int32, the second operand with a padded stride.
#pragma once
#include "vvcb_core.cuh"

namespace {

struct TrRom {                     // forward kernels M[k][n], int16, by type (0 DCT2, 1 DCT8, 2 DST7) and log2 size
  int16_t dct2[16 + 64 + 256 + 1024 + 4096];
  int16_t dct8[16 + 64 + 256 + 1024];
  int16_t dst7[16 + 64 + 256 + 1024];
  int32_t quantScales[12], invQuantScales[12];
  // low-frequency non-separable transform (CL/RomLFNST.cpp): kernels [4 sets][2][16 out][48 | 16 in], extended mode -> set,
  // and the diagonal order of a 4x4 group as x | y << 2
  int8_t  lfnst8[4 * 2 * 16 * 48], lfnst4[4 * 2 * 16 * 16];
  uint8_t lfnstLut[96], diag4[16];
};

// LFNST geometry of one job (TrQuant::xFwdLfnst / xInvLfnst, CL/TrQuant.cpp:316-560)
struct LfnstGeom {
  bool on, transpose;
  int sb, trSize, zeroOut;        // region side (4 or 8), inputs of the kernel (16 or 48), outputs kept (8 or 16)
  const int8_t* mat;              // [16][trSize]
};

__device__ __forceinline__ LfnstGeom make_lfnst(const TrRom& rom, int w, int h, int lw, int lh, bool ts, int lfnstIdx, int dirMode)
{
  LfnstGeom g;
  g.on = lfnstIdx > 0 && !ts;
  const bool whge3 = w >= 8 && h >= 8;
  g.sb = whge3 ? 8 : 4; g.trSize = whge3 ? 48 : 16;
  g.zeroOut = ((w == 4 && h == 4) || (w == 8 && h == 8)) ? 8 : 16;
  // PU::getWideAngIntraMode (CL/UnitTools.cpp:963-989) and TrQuant::getLFNSTIntraMode / getTransposeFlag (CL/TrQuant.cpp:288-312)
  int predMode = dirMode;
  if (dirMode >= 2) {
    const int delta = vabs(lw - lh);
    const int shift = delta == 0 ? 0 : delta == 1 ? 6 : delta == 2 ? 10 : delta == 3 ? 12 : delta == 4 ? 14 : 15;
    if (w > h && dirMode < 2 + shift) predMode += 65;
    else if (h > w && predMode > 66 - shift) predMode -= 67;
  }
  const int m = predMode < 0 ? predMode + 14 + 67 : (predMode >= 67 ? predMode + 14 : predMode);
  g.transpose = (m >= 67 + 14) || (m < 67 && m > 34);
  const int set = rom.lfnstLut[m];
  const int idx = vmax(lfnstIdx, 1) - 1;
  g.mat = whge3 ? rom.lfnst8 + (set * 2 + idx) * 16 * 48 : rom.lfnst4 + (set * 2 + idx) * 16 * 16;
  return g;
}

// position of region sample (x, y) in the LFNST input / output vector: row-major over the region without the bottom-right 4x4
// of an 8x8, column-major when transposed
__device__ __forceinline__ int lfnst_vec_index(const LfnstGeom& g, int x, int y)
{
  const int a = g.transpose ? y : x, b = g.transpose ? x : y;      // a runs fastest
  return g.sb == 4 ? b * 4 + a : (b < 4 ? b * 8 + a : 32 + (b - 4) * 4 + a);
}

// raster position (stride w) of the j-th entry of the LFNST scan: 4x4 groups (0,0), (0,1), (1,0) in diagonal order
__device__ __forceinline__ int lfnst_scan_pos(const TrRom& rom, int j, int w)
{
  const int g = j >> 4, d = rom.diag4[j & 15];
  const int x = (g == 2 ? 4 : 0) + (d & 3), y = (g == 1 ? 4 : 0) + (d >> 2);
  return y * w + x;
}

// A job is worked on by a TEAM of NT threads: the whole 128-thread CTA for large blocks, one warp (four jobs per CTA) for blocks of up
// to 256 samples, where 128 threads would mostly idle at barriers.
template <int NT> __device__ __forceinline__ int team_tid() { return NT == 32 ? (int)(threadIdx.x & 31) : (int)threadIdx.x; }
template <int NT> __device__ __forceinline__ void team_sync() { if (NT == 32) __syncwarp(); else __syncthreads(); }

// forward LFNST in place on the block A (stride w); tmp: 96 ints of scratch.  All threads of the team call it.
template <int NT>
__device__ __forceinline__ void lfnst_forward(const TrRom& rom, const LfnstGeom& g, int* A, int w, int* tmp)
{
  int* in = tmp; int* out = tmp + 48;
  const int tid = team_tid<NT>();
  team_sync<NT>();
  for (int t = tid; t < g.sb * g.sb; t += NT) {
    const int x = t % g.sb, y = t / g.sb;
    if (x < 4 || y < 4) in[lfnst_vec_index(g, x, y)] = A[y * w + x];
  }
  team_sync<NT>();
  for (int j = tid; j < g.trSize; j += NT) {
    int v = 0;
    if (j < g.zeroOut) {
      int acc = 0;
      for (int i = 0; i < g.trSize; i++) acc += in[i] * (int)g.mat[j * g.trSize + i];
      v = (acc + 64) >> 7;
    }
    out[j] = v;
  }
  team_sync<NT>();
  for (int j = tid; j < (g.sb == 4 ? 16 : 48); j += NT) A[lfnst_scan_pos(rom, j, w)] = out[j];
  team_sync<NT>();
}

// inverse LFNST in place (CL/TrQuant.cpp:262-286, 316-435)
template <int NT>
__device__ __forceinline__ void lfnst_inverse(const TrRom& rom, const LfnstGeom& g, int* A, int w, int* tmp)
{
  int* in = tmp; int* out = tmp + 48;
  const int tid = team_tid<NT>();
  team_sync<NT>();
  for (int i = tid; i < 16; i += NT) in[i] = A[lfnst_scan_pos(rom, i, w)];
  team_sync<NT>();
  for (int j = tid; j < g.trSize; j += NT) {
    int acc = 0;
    for (int i = 0; i < g.zeroOut; i++) acc += in[i] * (int)g.mat[i * g.trSize + j];
    out[j] = vmin(vmax((acc + 64) >> 7, -32768), 32767);
  }
  team_sync<NT>();
  for (int t = tid; t < g.sb * g.sb; t += NT) {
    const int x = t % g.sb, y = t / g.sb;
    if (x < 4 || y < 4) A[y * w + x] = out[lfnst_vec_index(g, x, y)];
  }
  team_sync<NT>();
}


__device__ __forceinline__ const int16_t* tr_kernel(const TrRom& rom, int type, int lg)
{
  const int off = lg == 2 ? 0 : lg == 3 ? 16 : lg == 4 ? 80 : lg == 5 ? 336 : 1360;
  return (type == 0 ? rom.dct2 : type == 1 ? rom.dct8 : rom.dst7) + off;
}

constexpr int kTuThreads = 128;

struct TuParams {
  const vvcb_tu_job* jobs;
  const int* list;     // indices of the jobs this launch works on
  int n;               // their number
  const int16_t* resi;
  const int16_t* pred;
  int32_t* coeff;      // optional
  int32_t* level;      // optional
  int16_t* reco;       // optional
  vvcb_tu_result* results;
  const int16_t* orig;
  int stride, bd;
  const TrRom* rom;
  // dependent quantisation runs between two passes of this kernel (vvcb_dq.cuh): pass 0 leaves the coefficients of those jobs
  // in dqCoeff, pass 1 picks their dequantised coefficients up from dqDeq and finishes (inverse, reconstruction, SSE)
  int32_t* dqCoeff;
  const int32_t* dqDeq;
  int phase;
  // optional explicit transform pair per job (intra sub-partitions, vvcb_isp_eval): VVCB_TR_* of the horizontal transform | vertical << 2,
  // read instead of mts_idx, which those jobs keep at 0 (implicit selection: no MTS zero-out or MTS rate semantics downstream)
  const uint8_t* trPair = nullptr;
};

__device__ __forceinline__ int clip16(int v) { return vmin(vmax(v, -32768), 32767); }

// team-wide sum of one value per thread (result valid in every thread)
template <int NT>
__device__ __forceinline__ long long team_sum(long long v, long long* red)
{
  for (int o = 16; o > 0; o >>= 1) {
    const int lo = __shfl_xor_sync(0xffffffffu, (int)(v & 0xffffffffll), o);
    const int hi = __shfl_xor_sync(0xffffffffu, (int)(v >> 32), o);
    v += ((long long)hi << 32) | (unsigned)lo;
  }
  if (NT == 32) return v;
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  long long t = 0;
  for (int i = 0; i < kTuThreads / 32; i++) t += red[i];
  return t;
}

constexpr int kTuSmallSamples = 256;      // blocks up to this size are worked on by one warp
constexpr int kTuSmallB = 288;            // their transposed intermediate: kept columns x (height + 1), largest for 32x8

// RESI: the reconstruction pass writes the inverse-transformed residual after its 16-bit clip into reco instead of the reconstruction, and
// takes no SSE (joint Cb-Cr, vvcb_chroma_joint_tu_eval: the residual is mapped to both components afterwards, and cannot be recovered
// from a clipped sample).  DCT-II jobs only.
template <int NT, bool RESI = false>
__global__ void __launch_bounds__(kTuThreads) tu_eval_kernel(TuParams P)
{
  constexpr int TEAMS = kTuThreads / NT;
  __shared__ int sA[NT == 32 ? TEAMS * kTuSmallSamples : 64 * 64];
  __shared__ int sB[NT == 32 ? TEAMS * kTuSmallB : 32 * 65];
  __shared__ long long red[kTuThreads / 32];
  const int team = NT == 32 ? (int)(threadIdx.x >> 5) : 0, tid = team_tid<NT>();
  int* A = sA + (NT == 32 ? team * kTuSmallSamples : 0);
  int* B = sB + (NT == 32 ? team * kTuSmallB : 0);
  const TrRom& rom = *P.rom;
  for (int q = blockIdx.x * TEAMS + team; q < P.n; q += gridDim.x * TEAMS) {
    const int ji = P.list[q];
    const vvcb_tu_job job = P.jobs[ji];
    const int lw = job.log2w, lh = job.log2h, w = 1 << lw, h = 1 << lh, n = w * h;
    const bool ts = job.mts_idx == 1;
    int hor = job.mts_idx > 1 ? (((job.mts_idx - 2) & 1) ? 1 : 2) : 0;
    int ver = job.mts_idx > 1 ? (((job.mts_idx - 2) >> 1) ? 1 : 2) : 0;
    if (P.trPair) { hor = P.trPair[ji] & 3; ver = P.trPair[ji] >> 2; }
    int wKeep = w - ((hor != 0 && w == 32) ? 16 : (w > 32 ? w - 32 : 0));
    int hKeep = h - ((ver != 0 && h == 32) ? 16 : (h > 32 ? h - 32 : 0));
    const LfnstGeom lf = make_lfnst(rom, w, h, lw, lh, ts, job.lfnst_idx, job.intra_mode);
    if (lf.on) {                                                   // only the LFNST region of primary coefficients exists (:853-867)
      if ((w == 4 && h > 4) || (w > 4 && h == 4)) { wKeep = 4; hKeep = 4; }
      else if (w >= 8 && h >= 8) { wKeep = 8; hKeep = 8; }
    }
    const int trShift = 15 - P.bd - ((lw + lh) >> 1);
    const int16_t* mh = tr_kernel(rom, hor, lw);
    const int16_t* mv = tr_kernel(rom, ver, lh);
    const int16_t* resi = P.resi + job.offset;
    const int hp = h + 1;
    // jobs whose quantiser is a kernel of its own (dependent quantisation, RDOQ for transform skip): vvcb_dq.cuh
    const bool dq = (job.flags & VVCB_TU_QUANT) && (job.flags & (VVCB_TU_DEPQUANT | VVCB_TU_RDOQ_TS));
    if (P.phase == 1 && !dq) continue;
    team_sync<NT>();
    if (P.phase == 1) {
      for (int i = tid; i < n; i += NT) A[i] = P.dqDeq[job.offset + i];
      team_sync<NT>();
    } else {
    for (int i = tid; i < n; i += NT) A[i] = ts ? ((int)resi[i] << trShift) : (int)resi[i];
    team_sync<NT>();
    if (!ts) {
      const int shift1 = lw + P.bd + 6 - 15, shift2 = lh + 6;
      const int add1 = shift1 > 0 ? 1 << (shift1 - 1) : 0, add2 = 1 << (shift2 - 1);
      for (int o = tid; o < wKeep * h; o += NT) {          // rows: B[k][j]
        const int k = o % wKeep, j = o / wKeep;
        const int16_t* m = mh + k * w;
        const int* a = A + j * w;
        int acc = 0;
        for (int t = 0; t < w; t++) acc += (int)m[t] * a[t];
        B[k * hp + j] = (acc + add1) >> shift1;
      }
      team_sync<NT>();
      for (int o = tid; o < n; o += NT) {                 // columns: A[l][k]
        const int k = o & (w - 1), l = o >> lw;
        int v = 0;
        if (k < wKeep && l < hKeep) {
          const int16_t* m = mv + l * h;
          const int* b = B + k * hp;
          int acc = 0;
          for (int t = 0; t < h; t++) acc += (int)m[t] * b[t];
          v = (acc + add2) >> shift2;
        }
        A[o] = v;
      }
      team_sync<NT>();
      if (lf.on) lfnst_forward<NT>(rom, lf, A, w, B);
    }
    }
    long long sumAbs = 0;
    if (P.phase == 0) {
      long long part = 0;
      for (int i = tid; i < n; i += NT) {
        part += vabs(A[i]);
        if (P.coeff) P.coeff[job.offset + i] = A[i];
        if (dq) P.dqCoeff[job.offset + i] = A[i];
      }
      sumAbs = team_sum<NT>(part, red);
      if (dq) {                                                          // the quantiser is another kernel: finish in pass 1
        if (tid == 0) {
          vvcb_tu_result r;
          r.abs_sum_coeff = (int)__dmul_rn((double)(int)sumAbs, ts && ((lw + lh) & 1) ? 1.0 / 1.414213562 : 1.0);   // CL/TrQuant.cpp:1098-1102
          r.abs_sum_level = 0; r.sse = 0; r.frac_bits = 0;
          P.results[ji] = r;
        }
        continue;
      }
    }
    int absLevel = 0;
    unsigned long long sse = 0;
    if (job.flags & VVCB_TU_QUANT) {
      const bool sqrtAdj = !ts && ((lw + lh) & 1);
      const int qScale = rom.quantScales[(sqrtAdj ? 6 : 0) + job.qp_rem];
      const int iScale = rom.invQuantScales[(sqrtAdj ? 6 : 0) + job.qp_rem];
      const int qbits = 14 + job.qp_per + trShift + (sqrtAdj ? -1 : 0);
      const long long qadd = 171ll << (qbits - 9);
      const int rightShift = 6 - (trShift + (sqrtAdj ? -1 : 0) + job.qp_per);
      const int tgt = vmin(16, 32 + rightShift - 7);
      const int inMin = -(1 << (tgt - 1)), inMax = (1 << (tgt - 1)) - 1;
      long long lpart = 0;
      if (P.phase == 0)
      for (int i = tid; i < n; i += NT) {
        const int c = A[i];
        const long long t = (long long)vabs(c) * qScale;
        const int mag = (int)((t + qadd) >> qbits);
        const int q = clip16(c < 0 ? -mag : mag);
        lpart += mag;
        if (P.level) P.level[job.offset + i] = q;
        const int qc = vmin(vmax(q, inMin), inMax);
        int d;
        if (rightShift > 0) d = (qc * iScale + (1 << (rightShift - 1))) >> rightShift;
        else                d = (int)((unsigned)(qc * iScale) << (-rightShift));
        A[i] = clip16(d);
      }
      absLevel = (int)team_sum<NT>(lpart, red);
      team_sync<NT>();                                     // A[] written per lane above, read across lanes below (the warp-team sum only shuffles)
      const int16_t* pred = P.pred + job.offset;
      const int16_t* org = P.orig + (size_t)job.y * P.stride + job.x;
      const int maxv = (1 << P.bd) - 1;
      long long spart = 0;
      if (!ts) {
        const int shift2 = 20 - P.bd;
        if (lf.on) lfnst_inverse<NT>(rom, lf, A, w, B);
        for (int o = tid; o < wKeep * h; o += NT) {        // columns first: B[j][y]
          const int j = o % wKeep, y = o / wKeep;
          int acc = 0;
          for (int k = 0; k < hKeep; k++) acc += (int)mv[k * h + y] * A[k * w + j];
          B[j * hp + y] = clip16((acc + 64) >> 7);
        }
        team_sync<NT>();
        for (int o = tid; o < n; o += NT) {               // rows
          const int x = o & (w - 1), y = o >> lw;
          int acc = 0;
          for (int k = 0; k < wKeep; k++) acc += (int)mh[k * w + x] * B[k * hp + y];
          const int r = clip16((acc + (1 << (shift2 - 1))) >> shift2);
          if (RESI) { P.reco[job.offset + o] = (int16_t)r; continue; }
          const int rec = vmin(vmax((int)pred[o] + (int)(int16_t)r, 0), maxv);
          if (P.reco) P.reco[job.offset + o] = (int16_t)rec;
          const int d = (int)org[y * P.stride + x] - rec;
          spart += (long long)d * d;
        }
      } else {
        const int off = trShift == 0 ? 0 : 1 << (trShift - 1);
        for (int o = tid; o < n; o += NT) {
          const int x = o & (w - 1), y = o >> lw;
          const int r = (int)(int16_t)((A[o] + off) >> trShift);
          const int rec = vmin(vmax((int)pred[o] + r, 0), maxv);
          if (P.reco) P.reco[job.offset + o] = (int16_t)rec;
          const int d = (int)org[y * P.stride + x] - rec;
          spart += (long long)d * d;
        }
      }
      sse = (unsigned long long)team_sum<NT>(spart, red);
    }
    if (P.phase == 1) {
      if (tid == 0) P.results[ji].sse = sse;
      continue;
    }
    if (tid == 0) {
      double scale = 1.0;
      if (ts && ((lw + lh) & 1)) scale = 1.0 / 1.414213562;               // CL/TrQuant.cpp:1098-1102
      vvcb_tu_result r;
      r.abs_sum_coeff = (int)__dmul_rn((double)(int)sumAbs, scale);
      r.abs_sum_level = absLevel;
      r.sse = sse;
      r.frac_bits = 0;
      P.results[ji] = r;
    }
  }
}

}  // namespace
