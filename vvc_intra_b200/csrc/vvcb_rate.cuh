// vvc_intra_b200 -- residual rate estimation kernel (sm_100a): the fractional bits CABACWriter::residual_coding( tu, COMPONENT_Y )
// adds on the reference's bit estimator (EL/CABACWriter.cpp:3773-3895, mts_coding :3897, last_sig_coeff :3960, residual_coding_subblock
// :4164, residual_codingTS :4025, residual_coding_subblockTS :4305; contexts CL/ContextModelling.h; BinProbModel_Std CL/Contexts.h:90-163;
// bypass / Golomb-Rice pricing EL/BinEncoder.cpp).  Every context-coded bin is priced from the model's current state and then adapts the
// model, so a TU is one serial chain over its bins: one warp per TU -- 32 lanes prepare, one lane walks -- on a private copy of the context
// models (the host sorts the jobs by size).  Luma, no sign hiding (off with dependent quantisation), no BDPCM, no ISP.
#pragma once
#include "vvcb_dq.cuh"

namespace {

struct RateRom { uint32_t binFracBits[512]; };     // ProbModelTables::m_binFracBits (CL/Contexts.cpp:57): [state][bin]

struct RateParams {
  const vvcb_tu_job* jobs;
  const int* order;          // indices of the VVCB_TU_RATE jobs, largest TU first
  int n;
  const int32_t* level;      // final levels, dense per job at job.offset
  vvcb_tu_result* results;   // frac_bits is written here
  const vvcb_ctx_states* states;         // the chroma instantiation reads vvcb_chroma_ctx_states here (and in statesOut)
  const DqRom* rom;
  const RateRom* rate;
  int depQuant;              // slice->getDepQuantEnabledFlag(): selects the state machine that picks the significance context set
  vvcb_ctx_states* statesOut = nullptr;   // optional: statesOut[job index] receives the models as the TU has left them (unchanged for an all-zero
                                          // TU); may be `states` itself when every job has a rate_idx of its own (vvcb_isp_eval)
};

struct RateEst {
  unsigned long long bits;
  const uint32_t* frac;      // binFracBits, staged in shared memory
};

// a context model as the kernel keeps it in shared memory: one 8-byte word per model
struct RateModel { uint32_t st; uint32_t rate; };     // st = state[0] | state[1] << 16

// flat model indices: the position of each context array inside vvcb_ctx_states, in models
#define VVCB_MODEL_AT(field) ((int)(offsetof(vvcb_ctx_states, field) / sizeof(vvcb_bin_model)))
constexpr int kMdlMts = VVCB_MODEL_AT(mts_idx), kMdlSigSbb = VVCB_MODEL_AT(sig_sbb), kMdlSig = VVCB_MODEL_AT(sig), kMdlPar = VVCB_MODEL_AT(par),
              kMdlGt1 = VVCB_MODEL_AT(gt1), kMdlGt2 = VVCB_MODEL_AT(gt2), kMdlLastX = VVCB_MODEL_AT(last_x), kMdlLastY = VVCB_MODEL_AT(last_y),
              kMdlTsSigSbb = VVCB_MODEL_AT(ts_sig_sbb), kMdlTsSig = VVCB_MODEL_AT(ts_sig), kMdlTsPar = VVCB_MODEL_AT(ts_par),
              kMdlTsGtx = VVCB_MODEL_AT(ts_gtx), kMdlTsLrg1 = VVCB_MODEL_AT(ts_lrg1), kMdlTsSign = VVCB_MODEL_AT(ts_sign);
#undef VVCB_MODEL_AT
constexpr int kRateModels = (int)(sizeof(vvcb_ctx_states) / sizeof(vvcb_bin_model));
static_assert(sizeof(vvcb_ctx_states) == kRateModels * sizeof(vvcb_bin_model) && sizeof(vvcb_bin_model) == 6, "vvcb_ctx_states is an array of 6-byte models");
// the same for the chroma models (vvcb_chroma_tu_eval)
#define VVCB_CMODEL_AT(field) ((int)(offsetof(vvcb_chroma_ctx_states, field) / sizeof(vvcb_bin_model)))
constexpr int kCMdlCbfCb = VVCB_CMODEL_AT(cbf_cb), kCMdlCbfCr = VVCB_CMODEL_AT(cbf_cr), kCMdlSigSbb = VVCB_CMODEL_AT(sig_sbb),
              kCMdlSig = VVCB_CMODEL_AT(sig), kCMdlPar = VVCB_CMODEL_AT(par), kCMdlGt1 = VVCB_CMODEL_AT(gt1), kCMdlGt2 = VVCB_CMODEL_AT(gt2),
              kCMdlLastX = VVCB_CMODEL_AT(last_x), kCMdlLastY = VVCB_CMODEL_AT(last_y);
#undef VVCB_CMODEL_AT
constexpr int kChromaRateModels = (int)(sizeof(vvcb_chroma_ctx_states) / sizeof(vvcb_bin_model));
static_assert(sizeof(vvcb_chroma_ctx_states) == kChromaRateModels * sizeof(vvcb_bin_model) && kChromaRateModels == 70, "vvcb_chroma_ctx_states is an array of 70 models");

// TBitEstimator::encodeBin: price, then BinProbModel_Std::update (MASK_0 0x7fe0, MASK_1 0x7ffe)
__device__ __forceinline__ void rate_bin(RateEst& e, RateModel* models, int ctx, unsigned bin)
{
  const uint2 m = *reinterpret_cast<const uint2*>(models + ctx);
  const unsigned rate0 = m.y >> 4, rate1 = m.y & 15;
  const unsigned s0 = m.x & 0xffffu, s1 = m.x >> 16;
  e.bits += e.frac[2 * ((s0 + s1) >> 8) + bin];
  unsigned n0 = s0 - ((s0 >> rate0) & 0x7fe0u), n1 = s1 - ((s1 >> rate1) & 0x7ffeu);
  if (bin) { n0 += (0x7fffu >> rate0) & 0x7fe0u; n1 += (0x7fffu >> rate1) & 0x7ffeu; }
  models[ctx].st = (n0 & 0xffffu) | (n1 << 16);
}

// BitEstimatorBase::encodeRemAbsEP with maxLog2TrDynamicRange 15
__device__ __forceinline__ void rate_rem_abs(RateEst& e, unsigned bins, unsigned rice)
{
  unsigned n;
  if (bins < (5u << rice)) n = (bins >> rice) + 1 + rice;
  else {
    unsigned prefix = 0, suffix;
    const unsigned code = (bins >> rice) - 5;
    if (code >= (1u << 12) - 1) { prefix = 12; suffix = 15; }
    else { while (code > (2u << prefix) - 2) prefix++; suffix = prefix + rice + 1; }
    n = 5 + prefix + suffix;
  }
  e.bits += (unsigned long long)n << 15;
}

constexpr int kRateWarps = 4;                        // TUs per CTA
constexpr int kRateThreads = 32 * kRateWarps;

// One warp per TU.  The chain over the bins cannot be cut (each bin adapts the model the next one of its context is priced from), but
// everything that feeds it can be prepared side by side: the 32 lanes find the last significant position, then derive for every scan
// position up to it ONE packed word -- the level, its context indices from the neighbourhood template and its Rice parameters -- into shared
// memory; lane 0 then walks that array in coding order against the TU's private copy of the context models (shared memory, one 8-byte word
// per model).  The walk touches no global memory apart from one sub-block position per sixteen coefficients.
//
// packed word, regular residual:  |level| (16) | significance context 0..11 (4) << 16 | greater-than context offset 1..20 (5) << 20 |
//                                 Rice parameter of a remainder after regular bins (2) << 25 | min(sum of the template, 31) (5) << 27
// packed word, transform skip:    modified level (17) | non-zero (1) << 17 | negative (1) << 18 | coded neighbours 0..2 (2) << 19 |
//                                 sign context 0..2 (2) << 21 | Rice parameter (2) << 23
// C: chroma (vvcb_chroma_ctx_states models, the chroma context derivations of H.266 9.3.4.2.5-9.3.4.2.8; chroma jobs never carry
// transform skip or MTS, so the mts_coding and transform-skip branches are not reached).
template <bool C = false>
__global__ void __launch_bounds__(kRateThreads) rate_kernel(RateParams P)
{
  __shared__ uint32_t sFrac[512];
  __shared__ RateModel sModels[kRateWarps][kRateModels];
  __shared__ uint32_t sInfo[kRateWarps][1024];
  for (int i = threadIdx.x; i < 512; i += blockDim.x) sFrac[i] = P.rate->binFracBits[i];
  __syncthreads();
  const DqRom& rom = *P.rom;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  RateModel* models = sModels[wib];
  uint32_t* info = sInfo[wib];
  for (int t = blockIdx.x * kRateWarps + wib; t < P.n; t += gridDim.x * kRateWarps) {
    const int ji = P.order[t];
    const vvcb_tu_job job = P.jobs[ji];
    const int lw = job.log2w, lh = job.log2h, w = 1 << lw, h = 1 << lh;
    const DqShape shp = rom.shape[lw - 2][lh - 2];
    const DqScanPos* scan = rom.pos + shp.first;
    const uint16_t* sbbPosTab = rom.sbbPos[lw - 2][lh - 2];
    const int32_t* coeff = P.level + job.offset;
    const int mts = job.mts_idx;

    // ---- the last significant scan position (the reference calls residual_coding only for a coded block)
    int scanPosLast = -1;
    for (int base = shp.numCoeff - 1; base >= 0 && scanPosLast < 0; base -= 128) {
      int idx[4], best = -1;
#pragma unroll
      for (int u = 0; u < 4; u++) { const int pos = base - 32 * u - lane; idx[u] = pos >= 0 ? (int)scan[pos].idx : -1; }
#pragma unroll
      for (int u = 3; u >= 0; u--) if (idx[u] >= 0 && coeff[idx[u]] != 0) best = base - 32 * u - lane;
      scanPosLast = __reduce_max_sync(0xffffffffu, best);
    }
    if (scanPosLast < 0) {
      if (lane == 0) P.results[ji].frac_bits = 0;
      if (P.statesOut) {
        const vvcb_bin_model* src = C ? reinterpret_cast<const vvcb_bin_model*>(P.states) + (size_t)job.rate_idx * kChromaRateModels
                                      : reinterpret_cast<const vvcb_bin_model*>(&P.states[job.rate_idx]);
        vvcb_bin_model* dst = C ? reinterpret_cast<vvcb_bin_model*>(P.statesOut) + (size_t)ji * kChromaRateModels
                                : reinterpret_cast<vvcb_bin_model*>(&P.statesOut[ji]);
        for (int i = lane; i < (C ? kChromaRateModels : kRateModels); i += 32) dst[i] = src[i];
      }
      continue;
    }

    {                                                            // this TU's private copy of the context models
      const vvcb_bin_model* src = C ? reinterpret_cast<const vvcb_bin_model*>(P.states) + (size_t)job.rate_idx * kChromaRateModels
                                    : reinterpret_cast<const vvcb_bin_model*>(&P.states[job.rate_idx]);
      for (int i = lane; i < (C ? kChromaRateModels : kRateModels); i += 32) {
        const vvcb_bin_model m = src[i];
        models[i].st = (uint32_t)m.state[0] | ((uint32_t)m.state[1] << 16);
        models[i].rate = m.rate;
      }
    }

    // ---- one packed word per scan position, all lanes
    unsigned long long sigGroups = 0;                           // by sub-block scan index
    const int prepEnd = mts == 1 ? shp.numCoeff - 1 : scanPosLast;
    for (int base = 0; base <= prepEnd; base += 32) {
      const int pos = base + lane;
      uint32_t word = 0;
      bool nz = false;
      if (pos <= prepEnd) {
        const DqScanPos sp = scan[pos];
        const int32_t* p = coeff + sp.idx;
        const int v = *p;
        nz = v != 0;
        if (mts == 1) {
          const int left = sp.x > 0 ? p[-1] : 0, above = sp.y > 0 ? p[-w] : 0;
          const int numPos = (left != 0) + (above != 0);
          int signCtx;
          if ((left == 0 && above == 0) || ((long long)left * above < 0)) signCtx = 0;
          else if (left >= 0 && above >= 0) signCtx = 1;
          else signCtx = 2;
          const int pred1 = vmax(vabs(left), vabs(above)), a = vabs(v);
          const int mod = a == pred1 ? 1 : (a < pred1 ? a + 1 : a);
          word = (uint32_t)mod | ((uint32_t)nz << 17) | ((uint32_t)(v < 0) << 18) | ((uint32_t)numPos << 19) | ((uint32_t)signCtx << 21) |
                 ((uint32_t)rom.tsRicePars[vmin(vabs(left) + vabs(above), 31)] << 23);
        } else {
          int sumAbs1 = 0, numPos = 0, sumAbs = 0;
#define VVCB_T(q) { const int a = vabs(q); sumAbs1 += vmin(4 + (a & 1), a); numPos += a != 0; sumAbs += a; }
          if (sp.x < w - 1) { VVCB_T(p[1]); if (sp.x < w - 2) VVCB_T(p[2]); if (sp.y < h - 1) VVCB_T(p[w + 1]); }
          if (sp.y < h - 1) { VVCB_T(p[w]); if (sp.y < h - 2) VVCB_T(p[2 * w]); }
#undef VVCB_T
          const int diag = sp.x + sp.y;
          const int sigCtx = vmin((sumAbs1 + 1) >> 1, 3) + (diag < 2 ? 4 : 0) + (!C && diag < 5 ? 4 : 0);
          const int ctxOff = vmin(sumAbs1 - numPos, 4) + 1 + (C ? (diag == 0 ? 5 : 0) : (diag == 0 ? 15 : diag < 3 ? 10 : diag < 10 ? 5 : 0));
          word = (uint32_t)vmin(vabs(v), 0xffff) | ((uint32_t)sigCtx << 16) | ((uint32_t)ctxOff << 20) |
                 ((uint32_t)rom.goRicePars[vmax(vmin(sumAbs - 20, 31), 0)] << 25) | ((uint32_t)vmin(sumAbs, 31) << 27);
        }
        info[pos] = word;
      }
      const unsigned b = __ballot_sync(0xffffffffu, nz);
      if (b & 0xffffu) sigGroups |= 1ull << (base >> 4);
      if (b >> 16) sigGroups |= 1ull << ((base >> 4) + 1);
    }
    __syncwarp();

    if (lane == 0) {
      RateEst e; e.bits = 0; e.frac = sFrac;
      const bool tsAllowed = (job.flags & VVCB_TU_TS_ALLOWED) != 0, mtsAllowed = (job.flags & VVCB_TU_MTS_ALLOWED) != 0;
      // ---- mts_coding
      if (tsAllowed) rate_bin(e, models, kMdlMts + 6, mts == 1);
      if (mts != 1 && mtsAllowed) {
        const unsigned symbol = mts != 0;
        rate_bin(e, models, kMdlMts, symbol);
        if (symbol)
          for (int i = 0, ctx = 7; i < 3; i++, ctx++) {
            const unsigned s2 = mts > i + 2;
            rate_bin(e, models, kMdlMts + ctx, s2);
            if (!s2) break;
          }
      }

      if (mts == 1) {
        // ---- residual_codingTS: forward over the sub-blocks, left / upper neighbours as context
        int remCtxBins = 2 * w * h;
        unsigned long long coded = 0;                           // m_sigCoeffGroupFlag, by raster position of the sub-block
        const int lastRaster = shp.numSbb - 1;
        for (int sb = 0; sb < shp.numSbb; sb++) {
          const int sbPos = sbbPosTab[sb], sy = sbPos / shp.widthInSbb, sx = sbPos - sy * shp.widthInSbb;
          const bool sig = (sigGroups >> sb) & 1;
          if (sig) coded |= 1ull << sbPos;
          const int sigLeft = sx > 0 ? (int)((coded >> (sbPos - 1)) & 1) : 0, sigAbove = sy > 0 ? (int)((coded >> (sbPos - shp.widthInSbb)) & 1) : 0;
          if (sb != shp.numSbb - 1 || (coded & ~(1ull << lastRaster)) != 0) {
            rate_bin(e, models, kMdlTsSigSbb + sigLeft + sigAbove, sig);
            if (!sig) continue;
          }
          const uint32_t* q = info + sb * 16;
          int numNonZero = 0;
          for (int i = 0; i < 16; i++) {
            const uint32_t x = q[i];
            const unsigned nzv = (x >> 17) & 1, numPos = (x >> 19) & 3;
            if (numNonZero || i != 15) { if (--remCtxBins >= 0) rate_bin(e, models, kMdlTsSig + numPos, nzv); else e.bits += 1ull << 15; }
            if (nzv) {
              if (--remCtxBins >= 0) rate_bin(e, models, kMdlTsSign + ((x >> 21) & 3), (x >> 18) & 1); else e.bits += 1ull << 15;
              numNonZero++;
              int rem = (int)(x & 0x1ffffu) - 1;
              if (--remCtxBins >= 0) rate_bin(e, models, kMdlTsLrg1 + numPos, rem != 0); else e.bits += 1ull << 15;
              if (rem) {
                rem -= 1;
                if (--remCtxBins >= 0) rate_bin(e, models, kMdlTsPar, rem & 1); else e.bits += 1ull << 15;
              }
            }
          }
          for (int i = 0; i < 16; i++) {
            const int mod = (int)(q[i] & 0x1ffffu);
            for (int k = 0, cutoff = 2; k < 4; k++, cutoff += 2)
              if (mod >= cutoff) { if (--remCtxBins >= 0) rate_bin(e, models, kMdlTsGtx + (cutoff >> 1), mod >= cutoff + 2); else e.bits += 1ull << 15; }
          }
          for (int i = 0; i < 16; i++) {
            const uint32_t x = q[i];
            const int mod = (int)(x & 0x1ffffu);
            if (mod >= 10) rate_rem_abs(e, (unsigned)(mod - 10) >> 1, (x >> 23) & 3);
          }
        }
        P.results[ji].frac_bits = e.bits;
      } else {
        // ---- last_sig_coeff
        {
          const DqScanPos lp = scan[scanPosLast];
          const int gX = rom.groupIdx[lp.x], gY = rom.groupIdx[lp.y];
          int maxX = rom.groupIdx[vmin(32, w) - 1], maxY = rom.groupIdx[vmin(32, h) - 1];
          if (mts > 1) { if (w == 32) maxX = rom.groupIdx[15]; if (h == 32) maxY = rom.groupIdx[15]; }
          const int offX = C ? 0 : lw == 2 ? 0 : lw == 3 ? 3 : lw == 4 ? 6 : lw == 5 ? 10 : 15, offY = C ? 0 : lh == 2 ? 0 : lh == 3 ? 3 : lh == 4 ? 6 : lh == 5 ? 10 : 15;
          const int shX = C ? vmin(2, w >> 3) : (lw + 1) >> 2, shY = C ? vmin(2, h >> 3) : (lh + 1) >> 2;
          const int mX = C ? kCMdlLastX : kMdlLastX, mY = C ? kCMdlLastY : kMdlLastY;
          for (int k = 0; k < gX; k++) rate_bin(e, models, mX + offX + (k >> shX), 1);
          if (gX < maxX) rate_bin(e, models, mX + offX + (gX >> shX), 0);
          for (int k = 0; k < gY; k++) rate_bin(e, models, mY + offY + (k >> shY), 1);
          if (gY < maxY) rate_bin(e, models, mY + offY + (gY >> shY), 0);
          if (gX > 3) e.bits += (unsigned long long)((gX - 2) >> 1) << 15;
          if (gY > 3) e.bits += (unsigned long long)((gY - 2) >> 1) << 15;
        }

        // ---- sub-blocks from the last significant one down to the DC one
        int regBins;
        {
          int tbW = w, tbH = h;
          if (mts > 1) { tbW = w == 32 ? 16 : w; tbH = h == 32 ? 16 : h; }
          regBins = (vmin(32, tbW) * vmin(32, tbH) * 28) >> 4;     // TU::getTbAreaAfterCoefZeroOut * 28 >> 4
        }
        const int stateTab = P.depQuant ? 32040 : 0;
        int state = 0;
        unsigned long long coded = 0;                              // by raster position
        for (int sb = scanPosLast >> 4; sb >= 0; sb--) {
          const int sbPos = sbbPosTab[sb], sy = sbPos / shp.widthInSbb, sx = sbPos - sy * shp.widthInSbb, minSub = sb * 16;
          const bool sig = (sigGroups >> sb) & 1, isLast = (scanPosLast >> 4) == sb;
          if (sig) coded |= 1ull << sbPos;
          if (mts > 1 && ((h == 32 && sy >= 4) || (w == 32 && sx >= 4))) continue;
          if (!isLast && sb != 0) {
            const int sigRight = sx + 1 < shp.widthInSbb ? (int)((coded >> (sbPos + 1)) & 1) : 0;
            const int sigLower = sy + 1 < shp.heightInSbb ? (int)((coded >> (sbPos + shp.widthInSbb)) & 1) : 0;
            rate_bin(e, models, (C ? kCMdlSigSbb : kMdlSigSbb) + (sigRight | sigLower), sig);
            if (!sig) continue;
          }
          const int firstSigPos = isLast ? scanPosLast : minSub + 15;
          int next = firstSigPos, numNonZero = 0, signBins = 0;
          const int inferSigPos = next != scanPosLast ? (sb != 0 ? minSub : -1) : next;
          for (; next >= minSub && regBins >= 4; next--) {
            const uint32_t x = info[next];
            const int a = (int)(x & 0xffffu);
            if (numNonZero || next != inferSigPos) {
              rate_bin(e, models, (C ? kCMdlSig + 8 * vmax(0, state - 1) : kMdlSig + 12 * vmax(0, state - 1)) + (int)((x >> 16) & 15), a != 0);
              regBins--;
            }
            if (a) {
              // ctxOffsetAbs(): template of this position, except for the TU's last position, whose significance context is never derived
              const int ctxOff = next != scanPosLast ? (int)((x >> 20) & 31) : 0;
              int rem = a - 1;
              numNonZero++; signBins++;
              rate_bin(e, models, (C ? kCMdlGt1 : kMdlGt1) + ctxOff, rem != 0);
              regBins--;
              if (rem) {
                rem -= 1;
                rate_bin(e, models, (C ? kCMdlPar : kMdlPar) + ctxOff, rem & 1);
                rem >>= 1;
                regBins--;
                rate_bin(e, models, (C ? kCMdlGt2 : kMdlGt2) + ctxOff, rem != 0);
                regBins--;
              }
            }
            state = (stateTab >> ((state << 2) + ((a & 1) << 1))) & 3;
          }
          const int firstPosMode2 = next;
          for (int i = firstSigPos; i >= minSub; i--) {
            const uint32_t x = info[i];
            const int a = (int)(x & 0xffffu);
            if (i > firstPosMode2) { if (a >= 4) rate_rem_abs(e, (unsigned)(a - 4) >> 1, (x >> 25) & 3); }   // 2nd pass: a remainder only from level 4 on
            else {                                                 // bypass-coded coefficient
              const int sumAll = (int)(x >> 27);
              const int pos0 = rom.goRiceZero[vmax(0, state - 1)][sumAll];
              rate_rem_abs(e, (unsigned)(a == 0 ? pos0 : (a <= pos0 ? a - 1 : a)), rom.goRicePars[sumAll]);
              state = (stateTab >> ((state << 2) + ((a & 1) << 1))) & 3;
              if (a) signBins++;
            }
          }
          e.bits += (unsigned long long)signBins << 15;
        }
        P.results[ji].frac_bits = e.bits;
      }
    }
    __syncwarp();
    if (P.statesOut) {
      vvcb_bin_model* dst = C ? reinterpret_cast<vvcb_bin_model*>(P.statesOut) + (size_t)ji * kChromaRateModels
                              : reinterpret_cast<vvcb_bin_model*>(&P.statesOut[ji]);
      for (int i = lane; i < (C ? kChromaRateModels : kRateModels); i += 32) {
        vvcb_bin_model m;
        m.state[0] = (uint16_t)(models[i].st & 0xffffu); m.state[1] = (uint16_t)(models[i].st >> 16);
        m.rate = (uint8_t)models[i].rate; m.pad = 0;
        dst[i] = m;
      }
      __syncwarp();
    }
  }
}

// vvcb_dq_rates (BinFracBits::intBits of each context, BinProbModel_Std::getFracBitsArray, CL/Contexts.h) of carried model states: the
// dependent quantiser of an ISP block is priced from the models as the previous block of its CU left them.  The two structs list the
// same contexts in the same order, vvcb_ctx_states with the MTS index contexts in front.  One thread per (snapshot, context).
constexpr int kDqRateModels = (int)(sizeof(vvcb_dq_rates) / (2 * sizeof(uint32_t)));
static_assert(kDqRateModels == kRateModels - 11, "vvcb_dq_rates lists the contexts of vvcb_ctx_states behind mts_idx[11]");

__global__ void __launch_bounds__(128) rates_from_states_kernel(const vvcb_ctx_states* states, int n, const RateRom* rom, vvcb_dq_rates* out)
{
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * kDqRateModels) return;
  const int s = (int)(t / kDqRateModels), i = (int)(t % kDqRateModels);
  const vvcb_bin_model m = reinterpret_cast<const vvcb_bin_model*>(&states[s])[11 + i];
  const int q = ((int)m.state[0] + (int)m.state[1]) >> 8;
  uint32_t* dst = reinterpret_cast<uint32_t*>(&out[s]) + 2 * i;
  dst[0] = rom->binFracBits[2 * q]; dst[1] = rom->binFracBits[2 * q + 1];
}

// The chroma models' prices in vvcb_dq_rates, for the chroma instantiation of dq_kernel: each chroma array at the start of its luma
// counterpart (sig_sbb[0..1], sig[set][0..7], par / gt1 / gt2[0..10], last_x / last_y[0..2]); dq_rate_kernel then derives the same
// DqRateTab layout, of which the chroma kernel reads those entries only.  One thread per (snapshot, residual context).
constexpr int kChromaResidualModels = kChromaRateModels - kCMdlSigSbb;

__global__ void __launch_bounds__(128) chroma_rates_from_states_kernel(const vvcb_chroma_ctx_states* states, int n, const RateRom* rom, vvcb_dq_rates* out)
{
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * kChromaResidualModels) return;
  const int s = (int)(t / kChromaResidualModels), i = kCMdlSigSbb + (int)(t % kChromaResidualModels);
  const vvcb_bin_model m = reinterpret_cast<const vvcb_bin_model*>(&states[s])[i];
  const int q = ((int)m.state[0] + (int)m.state[1]) >> 8;
  vvcb_dq_rates& r = out[s];
  uint32_t* dst = i < kCMdlSig ? r.sig_sbb[i - kCMdlSigSbb] : i < kCMdlPar ? r.sig[(i - kCMdlSig) >> 3][(i - kCMdlSig) & 7]
                : i < kCMdlGt1 ? r.par[i - kCMdlPar] : i < kCMdlGt2 ? r.gt1[i - kCMdlGt1] : i < kCMdlLastX ? r.gt2[i - kCMdlGt2]
                : i < kCMdlLastY ? r.last_x[i - kCMdlLastX] : r.last_y[i - kCMdlLastY];
  dst[0] = rom->binFracBits[2 * q]; dst[1] = rom->binFracBits[2 * q + 1];
}

}  // namespace
