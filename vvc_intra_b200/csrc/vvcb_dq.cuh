// vvc_intra_b200 -- dependent (trellis-coded) quantisation kernel (sm_100a).
//
// Reference behaviour: DQIntern::DepQuant::quant (CL/DepQuant.cpp:1592-1731) with its RateEstimator (:479-629), Quantizer
// (:694-844), State / CommonCtx (:895-1397), xDecide / xDecideAndUpdate (:1455-1589) and Quantizer::dequantBlock (:741-810);
// luma, flat scaling lists, the reference's compile-time switches as shipped (JVET_O0094 / O0052 / O0617 / O0256 on).
//
// Mapping.  The trellis is sequential in scan position and four states wide, so a TU is owned by a GROUP OF FOUR LANES
// (lane k = quantiser state k), eight TUs per warp.  All groups of a warp walk their scans in lock-step (the host sorts
// the jobs by size so that the groups of a warp have similar lengths); lanes exchange the three candidate costs of a
// state through shared memory.  The twelve states (current / previous / skip x 4) live in shared memory; the per-TU
// sub-block context memory (CommonCtx) and the decision trellis live in a global scratch slot owned by the group.
// After the forward pass lane 0 walks the trellis backwards, writes the levels and -- because the state a coefficient was
// quantised in is the `prevId` of its decision -- the dequantised coefficients in the same pass.
#pragma once
#include "vvcb_core.cuh"

namespace {

using namespace vvcb;

constexpr int kDqThreads = 128;
constexpr int kDqGroups  = kDqThreads / 4;
constexpr int kDqScaleBits = 15;
constexpr long long kDqHuge = 0x7fffffffffffffffll;
constexpr int kDqCtxBytes = 8 * (1024 + 64);                 // CommonCtx::m_memory for the largest TU
constexpr int kDqSlotBytes = kDqCtxBytes + 1024 * 16;        // + trellis: 4 packed decisions per scan position

// ---- read-only tables (built on the host at vvcb_create) ------------------------------------------------
struct DqScanPos {           // one scan position of one TU shape
  uint16_t idx;              // raster position (stride = TU width)
  uint8_t  x, y;
  uint16_t maxDist;          // NbInfoOut::maxDist (relative)
  uint8_t  numOut;           // neighbours outside the 4x4 sub-block ...
  uint8_t  pad;
  uint16_t outPos[5];        // ... relative to the first position of the sub-block
  uint16_t pad2;
};
struct DqShape { int first; int numCoeff, numSbb, widthInSbb, heightInSbb; };   // `first`: index of scan position 0 in DqRom::pos
struct DqRom {
  DqShape   shape[5][5];     // [log2w - 2][log2h - 2]
  DqScanPos pos[8464];       // all shapes back to back: (4 + 8 + 16 + 32 + 32)^2
  uint16_t  sbbPos[5][5][64];// sub-block scan -> raster position in the sub-block grid
  uint8_t   nbIn[16][6];     // inside-sub-block neighbours of an in-sub-block position: {num, inPos[5]} (shape independent)
  int32_t   goRiceBits[4][32];
  uint8_t   goRicePars[32], goRiceZero[3][32], groupIdx[32];
  uint8_t   tsRicePars[32];  // CoeffCodingContext::templateAbsSumTS (CL/ContextModelling.h:350-365)
  int32_t   quantScales[12], invQuantScales[12];
};

// per snapshot of context prices, derived once per call by dq_rate_kernel (RateEstimator::xSetGtxFlagBits etc.)
struct DqRateTab {
  int32_t gtx[21][6];
  int32_t sig[3][12][2];
  int32_t sigSbb[2][2];
};

struct alignas(16) DqState { // 96 bytes
  uint16_t  ctxInit[24];     // m_absLevelsAndCtxInit (first: copied as three 16-byte words)
  long long rdCost;
  int       numSigSbb, remRegBins, refSbbCtxId;
  int       sbbBits0, sbbBits1;
  int       sigCtx, gtxCtx;  // indices into DqRateTab::sig[set(stateId)] / gtx
  int       goRicePar, goRiceZero;
  int       pad;
};

struct DqGroupSmem {
  DqState   st[12];          // [set 0..2][state 0..3]; which set is current / previous / skip rotates
  long long cand[4][3];      // candidate costs A, Z, B of source state k
  long long pathCost[4];     // rdCost of the four decisions at scan position 0
  int32_t   lastX[12], lastY[12];   // ctxBits of RateEstimator::xSetLastCoeffOffset per group index
};

struct DqParams {
  const vvcb_tu_job* jobs;
  const int* order;          // DepQuant job indices sorted by first test position, longest scan first (dq_sort_kernel)
  const int* firstPos;       // first test position of order[i] (-1: nothing to quantise)
  int n;                     // number of DepQuant jobs
  const int32_t* coeff;      // forward-transform output (dense per job at job.offset)
  int32_t* level;            // out: levels (zero-filled by the caller)
  int32_t* deq;              // out: dequantised coefficients (zero-filled by the caller)
  vvcb_tu_result* results;   // abs_sum_level is written here
  const vvcb_dq_rates* rates;
  const DqRateTab* tabs;
  const DqRom* rom;
  uint8_t* scratch;          // kDqSlotBytes per group of the grid
  int bd;
  int sparse;                // 1: one TU per warp (group 0 works, the other seven idle) -- the latency-bound batches of a host walk
};

__global__ void dq_rate_kernel(const vvcb_dq_rates* rates, int n, DqRateTab* tabs)
{
  const int r = blockIdx.x;
  if (r >= n) return;
  const vvcb_dq_rates& c = rates[r];
  DqRateTab& t = tabs[r];
  for (int i = threadIdx.x; i < 21; i += blockDim.x) {
    const int par0 = (1 << kDqScaleBits) + (int)c.par[i][0], par1 = (1 << kDqScaleBits) + (int)c.par[i][1];
    t.gtx[i][0] = 0;
    t.gtx[i][1] = (int)c.gt1[i][0] + (1 << kDqScaleBits);
    t.gtx[i][2] = (int)c.gt1[i][1] + par0 + (int)c.gt2[i][0];
    t.gtx[i][3] = (int)c.gt1[i][1] + par1 + (int)c.gt2[i][0];
    t.gtx[i][4] = (int)c.gt1[i][1] + par0 + (int)c.gt2[i][1];
    t.gtx[i][5] = (int)c.gt1[i][1] + par1 + (int)c.gt2[i][1];
  }
  for (int i = threadIdx.x; i < 72; i += blockDim.x) (&t.sig[0][0][0])[i] = (int)(&c.sig[0][0][0])[i];
  for (int i = threadIdx.x; i < 4; i += blockDim.x) (&t.sigSbb[0][0])[i] = (int)(&c.sig_sbb[0][0])[i];
}

struct DqQuant {             // Quantizer::initQuantBlock, CL/DepQuant.cpp:694-739
  int qShift, maxQIdx, thres, distShift;
  long long qAdd, qScale, distAdd, distStepAdd, distOrgFact;
};

VHD int dq_ceil_log2(unsigned long long x)
{
  int n = 0;
  const int notPow2 = (x & (x - 1)) != 0;
  while (x > 1) { x >>= 1; n++; }
  return n + notPow2;
}

VHD DqQuant dq_init_quant(const DqRom& rom, int bd, int lw, int lh, int qp, double lambda)
{
  DqQuant q;
  const int qpDQ = qp + 1, qpPer = qpDQ / 6, qpRem = qpDQ - 6 * qpPer;
  const int nomShift = 15 - bd - ((lw + lh) >> 1);
  const int sqrt2 = (lw + lh) & 1;
  const int trShift = nomShift - sqrt2;
  const int invShift = 7 - qpPer - trShift;
  q.qShift = 13 + qpPer + trShift;
  q.qAdd = -((3ll << q.qShift) >> 1);
  q.qScale = rom.quantScales[sqrt2 * 6 + qpRem];
  q.maxQIdx = (1 << (vmin(16, 32 + invShift - 7) - 1)) - 4;
  q.thres = (int)((4ll << q.qShift) / (4 * q.qScale));           // thresLast / (4 * defaultQuantisationCoefficient), :1648-1656
  const int nomDShift = kDqScaleBits - 2 * nomShift + q.qShift + sqrt2;
  const double qScale2 = (double)(q.qScale * q.qScale);
  // the reference evaluates these in IEEE double without contraction; every product below is a single rounding
#if defined(__CUDA_ARCH__)
  const double den = __dmul_rn(qScale2, lambda);
  const double f = nomDShift < 0 ? __ddiv_rn(1.0, __dmul_rn((double)(1ll << (-nomDShift)), den)) : __ddiv_rn((double)(1ll << nomDShift), den);
  const long long pow2 = (long long)__dmul_rn(f, qScale2) + 1;
#else
  const double den = qScale2 * lambda;
  const double f = nomDShift < 0 ? 1.0 / ((double)(1ll << (-nomDShift)) * den) : (double)(1ll << nomDShift) / den;
  const long long pow2 = (long long)(f * qScale2) + 1;
#endif
  q.distShift = 62 + q.qShift - 30 - dq_ceil_log2((unsigned long long)pow2);
  q.distAdd = (1ll << q.distShift) >> 1;
#if defined(__CUDA_ARCH__)
  q.distStepAdd = (long long)__dadd_rn(__dmul_rn(f, (double)(1ll << (q.distShift + q.qShift))), .5);
  q.distOrgFact = (long long)__dadd_rn(__dmul_rn(f, (double)(1ll << (q.distShift + 1))), .5);
#else
  q.distStepAdd = (long long)(f * (double)(1ll << (q.distShift + q.qShift)) + .5);
  q.distOrgFact = (long long)(f * (double)(1ll << (q.distShift + 1)) + .5);
#endif
  return q;
}

// ---- first test position of every job (:1638-1662), one 4-lane group per job ---------------------------------
// jobsIdx: DepQuant job indices in any order; firstOut[i] belongs to jobsIdx[i]
__global__ void __launch_bounds__(kDqThreads) dq_first_kernel(const vvcb_tu_job* jobs, const int* jobsIdx, int n, const int32_t* coeffAll,
                                                              const DqRom* romp, int bd, int* firstOut)
{
  const DqRom& rom = *romp;
  const int k = threadIdx.x & 3;
  for (int base = blockIdx.x * kDqGroups; base < n; base += gridDim.x * kDqGroups) {
    const int i = base + (threadIdx.x >> 2);
    int firstTestPos = -1;
    if (i < n) {
      const vvcb_tu_job job = jobs[jobsIdx[i]];
      const int lw = job.log2w, lh = job.log2h, w = 1 << lw, h = 1 << lh;
      const DqShape shp = rom.shape[lw - 2][lh - 2];
      const DqScanPos* scan = rom.pos + shp.first;
      const int32_t* coeff = coeffAll + job.offset;
      const DqQuant Q = dq_init_quant(rom, bd, lw, lh, 6 * job.qp_per + job.qp_rem, job.lambda);
      const bool zeroOutTu = job.mts_idx > 1 && (w == 32 || h == 32);
      int start = shp.numCoeff - 1;                                 // positions past the 32x32 region are zero-out fillers
      if (job.lfnst_idx > 0) start = vmin(start, ((w == 4 && h == 4) || (w == 8 && h == 8)) ? 7 : 15);
      const int limX = (w == 32 && zeroOutTu) ? 16 : 32, limY = (h == 32 && zeroOutTu) ? 16 : 32;
      for (int s = start - k; s >= 0; s -= 4) {
        const DqScanPos sp = scan[s];
        if (sp.x >= limX || sp.y >= limY) continue;
        if (vabs(coeff[sp.idx]) > Q.thres) { firstTestPos = s; break; }
      }
    }
    firstTestPos = vmax(firstTestPos, __shfl_xor_sync(0xffffffffu, firstTestPos, 1));
    firstTestPos = vmax(firstTestPos, __shfl_xor_sync(0xffffffffu, firstTestPos, 2));
    if (i < n && k == 0) firstOut[i] = firstTestPos;
  }
}

// Counting sort of the jobs by first test position, longest scan first, so that the eight groups of a warp walk scans of the
// same length and reach their sub-block boundaries in the same iteration.  1025 bins; three launches: per-block histograms
// folded into a global one, a one-block exclusive scan over descending keys, and a scatter in which every block reserves its
// share of each bin with one global atomic and places its own elements with shared-memory atomics.
constexpr int kDqSortThreads = 256;
constexpr int kDqSortPerBlock = 4096;       // elements per block
constexpr int kDqBins = 1025;

__global__ void __launch_bounds__(kDqSortThreads) dq_hist_kernel(const int* firstIn, int n, int* binCount)
{
  __shared__ int bin[kDqBins];
  for (int i = threadIdx.x; i < kDqBins; i += blockDim.x) bin[i] = 0;
  __syncthreads();
  const int lo = blockIdx.x * kDqSortPerBlock, hi = vmin(n, lo + kDqSortPerBlock);
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(&bin[firstIn[i] + 1], 1);
  __syncthreads();
  for (int i = threadIdx.x; i < kDqBins; i += blockDim.x) if (bin[i]) atomicAdd(&binCount[i], bin[i]);
}

__global__ void dq_scan_kernel(int* binCount)      // in place: count -> first output index of the bin (descending keys)
{
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    int acc = 0;
    for (int b = kDqBins - 1; b >= 0; b--) { const int c = binCount[b]; binCount[b] = acc; acc += c; }
  }
}

__global__ void __launch_bounds__(kDqSortThreads) dq_scatter_kernel(const int* jobsIdx, const int* firstIn, int n, int* binCursor,
                                                                    int* orderOut, int* firstOut)
{
  __shared__ int bin[kDqBins], base[kDqBins];
  for (int i = threadIdx.x; i < kDqBins; i += blockDim.x) bin[i] = 0;
  __syncthreads();
  const int lo = blockIdx.x * kDqSortPerBlock, hi = vmin(n, lo + kDqSortPerBlock);
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) atomicAdd(&bin[firstIn[i] + 1], 1);
  __syncthreads();
  for (int i = threadIdx.x; i < kDqBins; i += blockDim.x) { base[i] = bin[i] ? atomicAdd(&binCursor[i], bin[i]) : 0; bin[i] = 0; }
  __syncthreads();
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    const int f = firstIn[i];
    const int at = base[f + 1] + atomicAdd(&bin[f + 1], 1);
    orderOut[at] = jobsIdx[i];
    firstOut[at] = f;
  }
}

// bits of an absolute level coded with regular bins under the state's greater-than contexts (:977-990)
__device__ __forceinline__ long long dq_level_bits(const DqRom& rom, const int32_t* gtx, int goRicePar, int absLevel)
{
  if (absLevel < 4) return gtx[absLevel];
  const unsigned value = (unsigned)(absLevel - 4) >> 1;
  return gtx[absLevel - (int)(value << 1)] + rom.goRiceBits[goRicePar][value < 32u ? value : 31u];
}

__device__ __forceinline__ uint32_t dq_pack(int absLevel, int prevId) { return (uint32_t)(absLevel & 0xffff) | ((uint32_t)(prevId + 2) << 16); }

#ifndef VVCB_DQ_MIN_CTAS
#define VVCB_DQ_MIN_CTAS 4
#endif
// C: chroma (vvcb_chroma_tu_eval): the chroma context sets and per-position offsets of H.266 9.3.4.2.5-9.3.4.2.8 -- significance offset
// d < 2 ? 4 : 0 into 8 contexts per state class, greater-than offset d == 0 ? 6 : 1, last-position contexts from the start of the chroma
// arrays with shift Clip3(0, 2, side >> 3) -- on prices laid out by chroma_rates_from_states_kernel (vvcb_rate.cuh).
template <bool C = false>
__global__ void __launch_bounds__(kDqThreads, VVCB_DQ_MIN_CTAS) dq_kernel(DqParams P)
{
  __shared__ DqGroupSmem smem[kDqGroups];
  const DqRom& rom = *P.rom;
  const int lane = threadIdx.x & 31, k = lane & 3;                 // k: this lane's quantiser state
  const int gInCta = threadIdx.x >> 2;
  DqGroupSmem& sm = smem[gInCta];
  const int slot = blockIdx.x * kDqGroups + gInCta;
  uint8_t* ctxMem = P.scratch + (size_t)slot * kDqSlotBytes;
  uint4* trellis = reinterpret_cast<uint4*>(ctxMem + kDqCtxBytes);
  const int groupsTotal = gridDim.x * kDqGroups;
  const int perRound = P.sparse ? groupsTotal >> 3 : groupsTotal;
  const int rounds = (P.n + perRound - 1) / perRound;

  for (int round = 0; round < rounds; round++) {
    // round-robin over the size-sorted job list: the 8 groups of a warp get neighbours in the sorted order
    const int ji = P.sparse ? ((lane >> 2) == 0 ? round * (groupsTotal >> 3) + (slot >> 3) : P.n) : round * groupsTotal + slot;
    const bool have = ji < P.n;
    vvcb_tu_job job;
    if (have) job = P.jobs[P.order[ji]];
    else { job.log2w = 2; job.log2h = 2; job.mts_idx = 0; job.offset = 0; job.qp_per = 4; job.qp_rem = 0; job.rate_idx = 0; job.lfnst_idx = 0; job.cbf_delta_bits = 0; job.lambda = 1.0; }
    const int lw = job.log2w, lh = job.log2h, w = 1 << lw, h = 1 << lh;
    const DqShape shp = rom.shape[lw - 2][lh - 2];
    const DqScanPos* scan = rom.pos + shp.first;
    const uint16_t* sbbPosTab = rom.sbbPos[lw - 2][lh - 2];
    const DqRateTab& tab = P.tabs[have ? job.rate_idx : 0];
    const int32_t* coeff = P.coeff + job.offset;
    const DqQuant Q = dq_init_quant(rom, P.bd, lw, lh, 6 * job.qp_per + job.qp_rem, job.lambda);
    int effW = w, effH = h;
    bool zeroOutTu = false;
    if (job.mts_idx > 1) { effH = h == 32 ? 16 : h; effW = w == 32 ? 16 : w; zeroOutTu = effH < h || effW < w; }
    const int regBinsInit = (vmin(32, effW) * vmin(32, effH) * 28) >> 4;
    const int sbbPad = (shp.numSbb + 15) & ~15;                    // the sub-block flags, padded so that the level arrays and the
    const int ctxStride = sbbPad + shp.numCoeff;                   // eight context sets stay 16-byte aligned (copied as uint4)

    const int firstTestPos = have ? P.firstPos[ji] : -1;           // dq_first_kernel, :1638-1662
    // The groups of a warp walk in lock-step from a COMMON start position, the warp's largest first test position rounded up to the end of
    // its sub-block; a group is idle until the walk reaches its own first test position.  All groups then cross their sub-block boundaries
    // -- the expensive step, State::updateStateEOS -- in the same iteration instead of one after the other.
    int top = firstTestPos;
    for (int o = 4; o < 32; o <<= 1) top = vmax(top, __shfl_xor_sync(0xffffffffu, top, o));
    const int startPos = top | 15, steps = top < 0 ? 0 : startPos + 1;
    const int lastFetch = vmax(firstTestPos, 0);

    // ---- init (:1665-1688)
    __syncwarp();
    for (int s = k; s < 12; s += 4) {
      DqState& st = sm.st[s];
      st.rdCost = kDqHuge >> 1;
      for (int i = 0; i < 24; i++) st.ctxInit[i] = 0;
      st.numSigSbb = 0; st.remRegBins = 4; st.refSbbCtxId = -1;
      st.sbbBits0 = 0; st.sbbBits1 = 0; st.sigCtx = 0; st.gtxCtx = 0; st.goRicePar = 0; st.goRiceZero = 0;
    }
    if (k < 2) {                                                   // RateEstimator::xSetLastCoeffOffset :541-567
      const int size = k ? h : w, lg = k ? lh : lw;
      const uint32_t (*ctx)[2] = k ? P.rates[job.rate_idx].last_y : P.rates[job.rate_idx].last_x;
      const int prefix = C ? 0 : lg == 2 ? 0 : lg == 3 ? 3 : lg == 4 ? 6 : lg == 5 ? 10 : 15;
      const int lastShift = C ? vmin(2, size >> 3) : (lg + 1) >> 2, bitOffset = k ? job.cbf_delta_bits : 0;
      const int maxCtxId = rom.groupIdx[vmin(32, size) - 1];
      int32_t* out = k ? sm.lastY : sm.lastX;
      uint32_t sum = 0;
      for (int c = 0; c < maxCtxId; c++) {
        const uint32_t* b = ctx[prefix + (c >> lastShift)];
        out[c] = (int32_t)(sum + b[0] + (c > 3 ? (uint32_t)((c - 2) >> 1) << kDqScaleBits : 0u) + (uint32_t)bitOffset);
        sum += b[1];
      }
      out[maxCtxId] = (int32_t)(sum + (maxCtxId > 3 ? (uint32_t)((maxCtxId - 2) >> 1) << kDqScaleBits : 0u) + (uint32_t)bitOffset);
    }
    __syncwarp();

    int curr = 0, prev = 1, skip = 2;          // which third of sm.st plays which role
    int currSet = 0, prevSet = 4;              // CommonCtx::m_currSbbCtx / m_prevSbbCtx
    const int32_t* sigTab = &tab.sig[vmax(k - 1, 0)][0][0];

    DqScanPos sp = scan[lastFetch];                                // this iteration's position; the next one is fetched a step ahead
    int coeffCur = coeff[sp.idx];
    for (int it = 0; it < steps; it++) {
      const int scanIdx = startPos - it;
      const DqScanPos nx = scan[vmin(vmax(scanIdx - 1, 0), lastFetch)];
      const int coeffNext = coeff[nx.idx];
      const bool act = scanIdx <= firstTestPos;                    // scanIdx >= 0 inside the loop
      { const int t = prev; prev = curr; curr = t; }               // std::swap(m_prevStates, m_currStates)
      long long dCost = kDqHuge >> 2;
      int dLevel = -1, dPrev = -2;
      int spt = 0, spX = 0, spY = 0;
      bool zeroOut = false;
      // Quantizer::preQuantCoeff :812-843 yields four candidates, quantisation indices q0 .. q0 + 3 filed under slot (index & 3).  A lane
      // needs two or three of them, so instead of building the table it evaluates the slot it wants: candidate i = (slot - q0) & 3.
      int q0 = 0;
      long long sAdd0 = 0;
      auto pq_level = [&](int slot) { return (q0 + ((slot - q0) & 3) + 1) >> 1; };
      auto pq_dist = [&](int slot) {
        const int i = (slot - q0) & 3;
        return ((sAdd0 + (long long)i * Q.distStepAdd) * (q0 + i) + Q.distAdd) >> Q.distShift;
      };
      if (act) {
        const int inside = scanIdx & 15;
        spX = sp.x; spY = sp.y;
        if (inside == 15 && scanIdx > 16 && scanIdx < shp.numCoeff - 1) spt = 1;                 // SCAN_SOCSBB
        else if (inside == 0 && scanIdx > 0 && scanIdx < shp.numCoeff - 16) spt = 2;             // SCAN_EOCSBB
        zeroOut = zeroOutTu && (sp.x >= effW || sp.y >= effH);
        if (!zeroOut) {
          const int absCoeff = vabs(coeffCur);
          const long long scaledOrg = (long long)absCoeff * Q.qScale;
          q0 = vmax(1, vmin(Q.maxQIdx, (int)((scaledOrg + Q.qAdd) >> Q.qShift)));
          sAdd0 = q0 * Q.distStepAdd - scaledOrg * Q.distOrgFact;
          // ---- State::checkRdCosts of previous state k :924-1049
          const DqState& ps = sm.st[prev * 4 + k];
          const int slotA = k < 2 ? 0 : 3, slotB = k < 2 ? 2 : 1;
          const int lvA = pq_level(slotA), lvB = pq_level(slotB);
          long long cA = ps.rdCost + pq_dist(slotA);
          long long cB = ps.rdCost + pq_dist(slotB);
          long long cZ = ps.rdCost;
          const int32_t* rice = rom.goRiceBits[ps.goRicePar];
          if (ps.remRegBins >= 4) {
            const int32_t* gtx = tab.gtx[ps.gtxCtx];
            const int sig0 = sigTab[ps.sigCtx * 2], sig1 = sigTab[ps.sigCtx * 2 + 1];
            cA += dq_level_bits(rom, gtx, ps.goRicePar, lvA);
            cB += dq_level_bits(rom, gtx, ps.goRicePar, lvB);
            if (spt == 0)      { cA += sig1; cB += sig1; cZ += sig0; }
            else if (spt == 1) { cA += ps.sbbBits1 + sig1; cB += ps.sbbBits1 + sig1; cZ += ps.sbbBits1 + sig0; }
            else if (ps.numSigSbb) { cA += sig1; cB += sig1; cZ += sig0; }
            else cZ = kDqHuge;                                     // "rdCostZ = decisionA.rdCost": can never win
          } else {
            cA += (1 << kDqScaleBits) + rice[lvA <= ps.goRiceZero ? lvA - 1 : (lvA < 32 ? lvA : 31)];
            cB += (1 << kDqScaleBits) + rice[lvB <= ps.goRiceZero ? lvB - 1 : (lvB < 32 ? lvB : 31)];
            cZ += rice[ps.goRiceZero];
          }
          sm.cand[k][0] = cA; sm.cand[k][1] = cZ; sm.cand[k][2] = cB;
        }
      }
      __syncwarp();
      if (act) {
        if (!zeroOut) {
          // decision d collects "A" and "Z" of source sA(d) and "B" of source sB(d): states 0/1 feed decisions 0/2, states 2/3 feed 1/3
          const int sA = k == 0 ? 0 : k == 1 ? 2 : k == 2 ? 1 : 3, sB = k == 0 ? 1 : k == 1 ? 3 : k == 2 ? 0 : 2;
          const int lvFromA = pq_level(sA < 2 ? 0 : 3);              // pqDataA of source sA
          const int lvFromB = pq_level(sB < 2 ? 2 : 1);              // pqDataB of source sB
          dCost = kDqHuge >> 2; dLevel = -1; dPrev = -2;
          // sources are visited in ascending order (xDecide :1474-1477), ties keep the earlier candidate
          if (sA < sB) {
            if (sm.cand[sA][0] < dCost) { dCost = sm.cand[sA][0]; dLevel = lvFromA; dPrev = sA; }
            if (sm.cand[sA][1] < dCost) { dCost = sm.cand[sA][1]; dLevel = 0; dPrev = sA; }
            if (sm.cand[sB][2] < dCost) { dCost = sm.cand[sB][2]; dLevel = lvFromB; dPrev = sB; }
          } else {
            if (sm.cand[sB][2] < dCost) { dCost = sm.cand[sB][2]; dLevel = lvFromB; dPrev = sB; }
            if (sm.cand[sA][0] < dCost) { dCost = sm.cand[sA][0]; dLevel = lvFromA; dPrev = sA; }
            if (sm.cand[sA][1] < dCost) { dCost = sm.cand[sA][1]; dLevel = 0; dPrev = sA; }
          }
          if (spt == 2) {                                            // checkRdCostSkipSbb :1068-1077
            const DqState& ss = sm.st[skip * 4 + k];
            const long long c = ss.rdCost + ss.sbbBits0;
            if (c < dCost) { dCost = c; dLevel = 0; dPrev = 4 + k; }
          }
          if ((k & 1) == 0) {                                        // checkRdCostStart :1051-1066, decisions 0 and 2
            const int lv = pq_level(k);                              // pqData[0] for decision 0, pqData[2] for decision 2
            const long long c = pq_dist(k) + sm.lastX[rom.groupIdx[spX]] + sm.lastY[rom.groupIdx[spY]] +
                                dq_level_bits(rom, tab.gtx[0], 0, lv);
            if (c < dCost) { dCost = c; dLevel = lv; dPrev = -1; }
          }
        } else if (spt == 2) {                                       // checkRdCostSkipSbbZeroOut :1079-1085
          const DqState& ss = sm.st[skip * 4 + k];
          dCost = ss.rdCost + ss.sbbBits0; dLevel = 0; dPrev = 4 + k;
        }
        // ---- the decision trellis (entries 4..7 of the reference are implied, see the backward pass)
        reinterpret_cast<uint32_t*>(trellis + scanIdx)[k] = dq_pack(dLevel, dPrev);
        if (scanIdx == 0) sm.pathCost[k] = dCost;                    // path costs at the end of the scan

        // ---- state update :1533-1588
        if (scanIdx) {
          DqState& cs = sm.st[curr * 4 + k];
          const int diag = nx.x + nx.y;
          const int sigOff = C ? (diag < 2 ? 4 : 0) : diag < 2 ? 8 : diag < 5 ? 4 : 0;
          const int gtxOff = C ? (diag < 1 ? 6 : 1) : diag < 1 ? 16 : diag < 3 ? 11 : diag < 10 ? 6 : 1;
          const int nextInside = (scanIdx - 1) & 15;
          if ((scanIdx & 15) == 0) {
            // ---- State::updateStateEOS :1275-1315 + CommonCtx::update :1317-1397 (after m_commonCtx.swap())
            const int cSet = prevSet, pSet = currSet;                // the sets after the swap
            cs.rdCost = dCost;
            if (dPrev > -2) {
              const DqState* pst = nullptr;
              if (dPrev >= 4)      { pst = &sm.st[skip * 4 + dPrev - 4]; cs.numSigSbb = 0; for (int i = 0; i < 8; i++) cs.ctxInit[i] = 0; }
              else if (dPrev >= 0) { pst = &sm.st[prev * 4 + dPrev]; cs.numSigSbb = pst->numSigSbb + (dLevel != 0); *reinterpret_cast<uint4*>(cs.ctxInit) = *reinterpret_cast<const uint4*>(pst->ctxInit); }
              else                 { cs.numSigSbb = 1; for (int i = 0; i < 8; i++) cs.ctxInit[i] = 0; }
              reinterpret_cast<uint8_t*>(cs.ctxInit)[0] = (uint8_t)vmin(255, dLevel);     // insidePos == 0
              uint8_t* sbbFlags = ctxMem + (size_t)(cSet + k) * ctxStride;
              uint8_t* levels = sbbFlags + sbbPad;
              // the copies run in 16-byte words; rounding the level window up only touches entries no template reads
              const int cpWords = (nx.maxDist + 15) >> 4, sbbWords = sbbPad >> 4;
              uint4* dstF = reinterpret_cast<uint4*>(sbbFlags);
              uint4* dstL = reinterpret_cast<uint4*>(levels + scanIdx);      // scanIdx is a multiple of 16 here
              if (pst && pst->refSbbCtxId >= 0) {
                const uint8_t* srcSet = ctxMem + (size_t)(pSet + pst->refSbbCtxId) * ctxStride;
                const uint4* srcF = reinterpret_cast<const uint4*>(srcSet);
                const uint4* srcL = reinterpret_cast<const uint4*>(srcSet + sbbPad + scanIdx);
                for (int i = 0; i < sbbWords; i++) dstF[i] = srcF[i];
                for (int i = 1; i < cpWords; i++) dstL[i] = srcL[i];           // word 0 is this sub-block, written below
              } else {
                const uint4 z = { 0u, 0u, 0u, 0u };
                for (int i = 0; i < sbbWords; i++) dstF[i] = z;
                for (int i = 1; i < cpWords; i++) dstL[i] = z;
              }
              sbbFlags[sbbPosTab[scanIdx >> 4]] = cs.numSigSbb != 0;
              dstL[0] = *reinterpret_cast<const uint4*>(cs.ctxInit);
              const int nsp = sbbPosTab[(scanIdx - 1) >> 4];
              const int ny = nsp / shp.widthInSbb, nxs = nsp - ny * shp.widthInSbb;
              const int right = nxs < shp.widthInSbb - 1 ? nsp + 1 : 0, below = ny < shp.heightInSbb - 1 ? nsp + shp.widthInSbb : 0;
              const int sigNSbb = ((right ? sbbFlags[right] : 0) || (below ? sbbFlags[below] : 0)) ? 1 : 0;
              cs.numSigSbb = 0;
              cs.remRegBins = pst ? pst->remRegBins : regBinsInit;
              cs.goRicePar = 0;
              cs.refSbbCtxId = k;
              cs.sbbBits0 = tab.sigSbb[sigNSbb][0]; cs.sbbBits1 = tab.sigSbb[sigNSbb][1];
              const int scanBeg = scanIdx - 16;
              const uint8_t* absLevels = levels + scanBeg;
#pragma unroll 4
              for (int id = 0; id < 16; id++) {
                const DqScanPos nb = scan[scanBeg + id];
                int sumAbs = 0, sumAbs1 = 0, sumNum = 0;
                // five predicated, independent loads (absent neighbours re-read entry 0 of the window and count as zero)
#pragma unroll
                for (int j = 0; j < 5; j++) {
                  const bool on = j < nb.numOut;
                  const int v = on ? absLevels[nb.outPos[j]] : 0;
                  sumAbs += v; sumAbs1 += vmin(4 + (v & 1), v); sumNum += v != 0;
                }
                cs.ctxInit[8 + id] = (uint16_t)(sumNum + (sumAbs1 << 3) + (vmin(127, sumAbs) << 8));
              }
              for (int i = 0; i < 8; i++) cs.ctxInit[i] = 0;
              const int tinit = cs.ctxInit[8 + nextInside];
              const int sumNum = tinit & 7, sumAbs1 = (tinit >> 3) & 31, sumGt1 = sumAbs1 - sumNum;
              cs.sigCtx = sigOff + vmin((sumAbs1 + 1) >> 1, 3);
              cs.gtxCtx = gtxOff + (sumGt1 < 4 ? sumGt1 : 4);
            }
          } else if (!zeroOut) {
            // ---- State::updateState<numIPos> :1109-1273
            cs.rdCost = dCost;
            if (dPrev > -2) {
              if (dPrev >= 0) {
                const DqState& pst = sm.st[prev * 4 + dPrev];
                cs.numSigSbb = pst.numSigSbb + (dLevel != 0);
                cs.refSbbCtxId = pst.refSbbCtxId;
                cs.sbbBits0 = pst.sbbBits0; cs.sbbBits1 = pst.sbbBits1;
                cs.remRegBins = pst.remRegBins - 1;
                cs.goRicePar = pst.goRicePar;
                if (cs.remRegBins >= 4) cs.remRegBins -= dLevel < 2 ? dLevel : 3;
#pragma unroll
                for (int i = 0; i < 3; i++) reinterpret_cast<uint4*>(cs.ctxInit)[i] = reinterpret_cast<const uint4*>(pst.ctxInit)[i];
              } else {
                cs.numSigSbb = 1; cs.refSbbCtxId = -1;
                cs.remRegBins = regBinsInit - (dLevel < 2 ? dLevel : 3);
                for (int i = 0; i < 24; i++) cs.ctxInit[i] = 0;
              }
              uint8_t* lv = reinterpret_cast<uint8_t*>(cs.ctxInit);
              lv[scanIdx & 15] = (uint8_t)vmin(255, dLevel);
              const uint8_t* nbIn = rom.nbIn[nextInside];
              const int tinit = cs.ctxInit[8 + nextInside];
              int sumAbs1 = (tinit >> 3) & 31, sumNum = tinit & 7, sumAbs = tinit >> 8;
              for (int j = 0; j < nbIn[0]; j++) {
                const int v = lv[nbIn[1 + j]];
                sumAbs1 += vmin(4 + (v & 1), v); sumNum += v != 0; sumAbs += v;
              }
              if (cs.remRegBins >= 4) {
                const int sumGt1 = sumAbs1 - sumNum;
                cs.sigCtx = sigOff + vmin((sumAbs1 + 1) >> 1, 3);
                cs.gtxCtx = gtxOff + (sumGt1 < 4 ? sumGt1 : 4);
                cs.goRicePar = rom.goRicePars[vmax(vmin(31, sumAbs - 20), 0)];
              } else {
                sumAbs = vmin(31, sumAbs);
                cs.goRicePar = rom.goRicePars[sumAbs];
                cs.goRiceZero = rom.goRiceZero[vmax(0, k - 1)][sumAbs];
              }
            }
          }
        }
      }
      // swaps shared by the four lanes of the group (uniform inside the group)
      if (act && scanIdx) {
        if ((scanIdx & 15) == 0) { const int t = currSet; currSet = prevSet; prevSet = t; }
        if (spt == 1) { const int t = prev; prev = skip; skip = t; }
      }
      sp = nx; coeffCur = coeffNext;
      __syncwarp();
    }

    // ---- best path (:1713-1722) and the backward pass (:1724-1731) fused with Quantizer::dequantBlock (:741-810)
    if (have && k == 0 && firstTestPos >= 0) {
      int prevId = -2;
      long long minPathCost = 0;
      for (int s = 0; s < 4; s++) if (sm.pathCost[s] < minPathCost) { prevId = s; minPathCost = sm.pathCost[s]; }
      const int qpDQ = 6 * job.qp_per + job.qp_rem + 1, qpPer = qpDQ / 6, qpRem = qpDQ - 6 * qpPer;
      const int sqrt2 = (lw + lh) & 1;
      const int shift = 7 - qpPer - (15 - P.bd - ((lw + lh) >> 1) - sqrt2);
      const int invScale = rom.invQuantScales[sqrt2 * 6 + qpRem];
      const long long scaleEff = shift < 0 ? (long long)invScale << -shift : invScale;   // the in-place `invQScale <<= -shift`
      const long long add = shift < 0 ? 0 : ((1ll << shift) >> 1);
      int absSum = 0;
      // four positions per round: their trellis words, scan entries and coefficients are fetched together (independent
      // loads), then the chain is resolved in registers
      const int lastPos = shp.numCoeff - 1;
      for (int s0 = 0; prevId >= 0; s0 += 4) {
        uint4 e[4]; int idx[4], cf[4];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          const int s = vmin(s0 + i, lastPos);
          e[i] = trellis[s];
          idx[i] = scan[s].idx;
        }
#pragma unroll
        for (int i = 0; i < 4; i++) cf[i] = coeff[idx[i]];
#pragma unroll
        for (int i = 0; i < 4; i++) {
          if (prevId < 0) break;
          const int scanIdx = s0 + i;
          int absLevel;
          if (prevId >= 4 && (scanIdx & 15) != 0) absLevel = 0;      // inside a skipped sub-block: {level 0, prevId unchanged}
          else {
            const int d = prevId & 3;                                // at eosbb entries 4..7 == 0..3
            const uint32_t w = d == 0 ? e[i].x : d == 1 ? e[i].y : d == 2 ? e[i].z : e[i].w;
            absLevel = (int)(w & 0xffff);
            prevId = (int)(w >> 16) - 2;
          }
          if (absLevel) {
            const bool neg = cf[i] < 0;
            const int state = prevId < 0 ? 0 : (prevId & 3);         // the state this coefficient was quantised in
            P.level[job.offset + idx[i]] = neg ? -absLevel : absLevel;
            const long long qIdx = 2ll * absLevel - (state >> 1);
            long long nom = ((neg ? -qIdx : qIdx) * scaleEff + add) >> (shift < 0 ? 0 : shift);
            nom = nom < -32768 ? -32768 : (nom > 32767 ? 32767 : nom);
            P.deq[job.offset + idx[i]] = (int32_t)nom;
            absSum += absLevel;
          }
        }
      }
      P.results[P.order[ji]].abs_sum_level = absSum;
    }
    __syncwarp();
  }
}

// =====================================================================================================
// RDOQ of transform-skip blocks: QuantRDOQ::xRateDistOptQuantTS (CL/QuantRDOQ.cpp:1243-1485) with xGetCodedLevelTSPred
// (:2000-2065), xGetICRateTS (:2067-2150), xGetErrScaleCoeff (:383-393) and the transform-skip contexts of
// CoeffCodingContext (CL/ContextModelling.h:197-365).  The decision of a coefficient depends on the decided levels of its
// left and upper neighbours and on the sub-block flags before it, so a block is one serial chain: one warp per block (32
// lanes stage, one walks).  Costs are IEEE doubles combined in the reference's order (no contraction).
// =====================================================================================================
struct RdoqParams {
  const vvcb_tu_job* jobs;
  const int* order;          // RDOQ job indices, largest block first
  int n;
  const int32_t* coeff;      // transform-skip coefficients (residual << transformShift), dense per job at job.offset
  int32_t* level;            // out (zero-filled by the caller)
  int32_t* deq;              // out: dequantised coefficients, Quant::dequant (CL/Quant.cpp:423-540)
  vvcb_tu_result* results;
  const vvcb_dq_rates* rates;
  const DqRom* rom;
  int bd;
};

// the transform-skip prices of one vvcb_dq_rates snapshot, as the kernel stages them in shared memory
struct TsRates { uint32_t sig_sbb[3][2], sig[3][2], par[1][2], gtx[5][2], lrg1[4][2], sign[6][2]; };
static_assert(sizeof(vvcb_dq_rates) - offsetof(vvcb_dq_rates, ts_sig_sbb) >= sizeof(TsRates) &&
              offsetof(vvcb_dq_rates, ts_sign) - offsetof(vvcb_dq_rates, ts_sig_sbb) == offsetof(TsRates, sign), "TsRates mirrors the tail of vvcb_dq_rates");

__device__ __forceinline__ int rdoq_ic_rate_ts(int absLevel, const TsRates& r, const uint32_t* sign, const uint32_t* gt1, int sgn, int ricePar)
{
  int rate = (int)sign[sgn];
  if (absLevel > 1) {
    rate += (int)gt1[1];
    rate += (int)r.par[0][(absLevel - 2) & 1];
    int cutoff = 2;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      if (absLevel >= cutoff) rate += (int)r.gtx[cutoff >> 1][absLevel >= cutoff + 2];
      cutoff += 2;
    }
    if (absLevel >= cutoff) {
      unsigned symbol = (unsigned)(absLevel - cutoff) >> 1, length;
      if (symbol < (5u << ricePar)) {
        length = symbol >> ricePar;
        rate += (int)((length + 1 + ricePar) << kDqScaleBits);
      } else {
        length = (unsigned)ricePar;
        symbol -= 5u << ricePar;
        while (symbol >= (1u << length)) symbol -= 1u << (length++);
        rate += (int)((5 + length + 1 - ricePar + length) << kDqScaleBits);
      }
    }
  } else if (absLevel == 1) rate += (int)gt1[0];
  else rate = 0;
  return rate;
}

constexpr int kTsWarps = 4;                          // blocks per CTA
constexpr int kTsThreads = 32 * kTsWarps;

// One warp per block: the 32 lanes stage the scan, the scaled magnitudes and the prices in shared memory, lane 0 walks the chain there
// (the decided levels of the left / upper neighbours are read back from a shared-memory raster), global memory sees only the results.
__global__ void __launch_bounds__(kTsThreads) rdoq_ts_kernel(RdoqParams P)
{
  __shared__ TsRates sRates[kTsWarps];
  __shared__ uint32_t sScan[kTsWarps][1024];         // raster index | x << 16 | y << 24, by scan position
  __shared__ uint32_t sMag[kTsWarps][1024];          // levelDouble | (coefficient < 0) << 31, by scan position
  __shared__ int16_t sLevel[kTsWarps][1024];         // decided levels, raster
  const DqRom& rom = *P.rom;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  for (int t = blockIdx.x * kTsWarps + wib; t < P.n; t += gridDim.x * kTsWarps) {
    const int ji = P.order[t];
    const vvcb_tu_job job = P.jobs[ji];
    const int lw = job.log2w, lh = job.log2h, w = 1 << lw;
    const DqShape shp = rom.shape[lw - 2][lh - 2];
    const DqScanPos* scan = rom.pos + shp.first;
    const uint16_t* sbbPosTab = rom.sbbPos[lw - 2][lh - 2];
    const int32_t* coeff = P.coeff + job.offset;
    int32_t* level = P.level + job.offset;
    int32_t* deq = P.deq + job.offset;
    const double lambda = job.lambda;
    const int trShift = 15 - P.bd - ((lw + lh) >> 1);
    const int qBits = 14 + job.qp_per + trShift;
    const int quantCoeff = rom.quantScales[job.qp_rem];
    const TsRates& R = sRates[wib];
    uint32_t* scn = sScan[wib];
    uint32_t* mag = sMag[wib];
    int16_t* lvl = sLevel[wib];
    {
      const uint32_t* src = &P.rates[job.rate_idx].ts_sig_sbb[0][0];
      for (int i = lane; i < (int)(sizeof(TsRates) / 4); i += 32) reinterpret_cast<uint32_t*>(&sRates[wib])[i] = src[i];
      const long long cap = 0x7fffffffll - (1ll << (qBits - 1));
      for (int pos = lane; pos < shp.numCoeff; pos += 32) {
        const DqScanPos sp = scan[pos];
        const int c = coeff[sp.idx];
        const long long tmpLevel = (long long)vabs(c) * quantCoeff;
        scn[pos] = (uint32_t)sp.idx | ((uint32_t)sp.x << 16) | ((uint32_t)sp.y << 24);
        mag[pos] = (uint32_t)(tmpLevel < cap ? tmpLevel : cap) | (c < 0 ? 0x80000000u : 0u);
        lvl[pos] = 0;                                  // numCoeff == w * h for a transform-skip block
      }
    }
    __syncwarp();
    if (lane == 0) {
      // xGetErrScaleCoeff: 2^15 * 2^(-2 transformShift) / QStep / QStep
      const double errorScale = __ddiv_rn(__ddiv_rn(ldexp(32768.0, -2 * trShift), (double)quantCoeff), (double)quantCoeff);
      const int iScale = rom.invQuantScales[job.qp_rem];
      const int rightShift = 6 - (trShift + job.qp_per);
      const int tgt = vmin(16, 32 + rightShift - 7);
      const int inMin = -(1 << (tgt - 1)), inMax = (1 << (tgt - 1)) - 1;
      unsigned long long sigGroups = 0;                 // m_sigCoeffGroupFlag, by raster position of the sub-block
      bool anySigCG = false;
      int absSum = 0;
      for (int sb = 0; sb < shp.numSbb; sb++) {
        const int sbPos = sbbPosTab[sb];
        const int sy = sbPos / shp.widthInSbb, sx = sbPos - sy * shp.widthInSbb;
        const int sigLeft = sx > 0 ? (int)((sigGroups >> (sbPos - 1)) & 1) : 0;
        const int sigAbove = sy > 0 ? (int)((sigGroups >> (sbPos - shp.widthInSbb)) & 1) : 0;
        const uint32_t* bitsSigGroup = R.sig_sbb[sigLeft + sigAbove];
        int noCoeffCoded = 0;
        bool sig = false;
        double baseCost = 0.0, sigCostSum = 0.0, codedLevelAndDist = 0.0, uncodedDist = 0.0;
        for (int i = 0; i < 16; i++) {
          const uint32_t sc = scn[sb * 16 + i], mg = mag[sb * 16 + i];
          const int blk = (int)(sc & 0xffffu), spx = (int)((sc >> 16) & 0xff), spy = (int)(sc >> 24);
          const int levelDouble = (int)(mg & 0x7fffffffu), sgn = (int)(mg >> 31);
          const int roundAbs = vmin(32767, (int)(((long long)levelDouble + (1ll << (qBits - 1))) >> qBits));
          const int minAbs = roundAbs > 1 ? roundAbs - 1 : 1;
          const int upAbs = vmin(32767, vmin(32767, levelDouble >> qBits) + 1);
          const int right = spx > 0 ? (int)lvl[blk - 1] : 0;      // neighTS: left ...
          const int below = spy > 0 ? (int)lvl[blk - w] : 0;      // ... and upper neighbour
          const int pred1 = vmax(vabs(below), vabs(right));
          int tested[3], nTested = 0;
          tested[nTested++] = roundAbs;
          if (minAbs != roundAbs) tested[nTested++] = minAbs;
          const int predPixel = upAbs == pred1 ? 1 : (upAbs < pred1 ? upAbs + 1 : upAbs);
          if (upAbs != roundAbs && upAbs != minAbs && predPixel == 1) tested[nTested++] = upAbs;
          const double dErr = (double)levelDouble;
          const double cost0 = __dmul_rn(__dmul_rn(dErr, dErr), errorScale);
          const int numPos = (right != 0) + (below != 0);
          const uint32_t* bitsSig = R.sig[numPos];
          const int ricePar = rom.tsRicePars[vmin(vabs(right) + vabs(below), 31)];
          int signCtx;
          if ((right == 0 && below == 0) || ((long long)right * below < 0)) signCtx = 0;
          else if (right >= 0 && below >= 0) signCtx = 1;
          else signCtx = 2;
          const uint32_t* bitsSign = R.sign[signCtx];
          const uint32_t* bitsGt1 = R.lrg1[numPos];
          const bool isLast = i == 15 && noCoeffCoded == 0;
          // xGetCodedLevelTSPred
          double cost, csig = 0.0, currCostSig = 0.0;
          int best = 0;
          bool done = false;
          if (!isLast && tested[0] < 3) {
            csig = __dmul_rn(lambda, (double)bitsSig[0]);
            cost = __dadd_rn(cost0, csig);
            done = tested[0] == 0;
          } else cost = 1.7976931348623157e308;
          if (!done) {
            if (!isLast) currCostSig = __dmul_rn(lambda, (double)bitsSig[1]);
            for (int k = 0; k < nTested; k++) {
              const int absLevel = tested[k];
              const double e = (double)(levelDouble - (int)((unsigned)absLevel << qBits));
              const double err = __dmul_rn(__dmul_rn(e, e), errorScale);
              const int mod = absLevel == pred1 ? 1 : (absLevel < pred1 ? absLevel + 1 : absLevel);
              double cur = __dadd_rn(err, __dmul_rn(lambda, (double)rdoq_ic_rate_ts(mod, R, bitsSign, bitsGt1, sgn, ricePar)));
              cur = __dadd_rn(cur, currCostSig);
              if (cur < cost) { best = absLevel; cost = cur; csig = currCostSig; }
            }
          }
          if (best > 0) noCoeffCoded++;
          const int lv = (best != 0 && sgn) ? -best : best;
          lvl[blk] = (int16_t)lv;
          baseCost = __dadd_rn(baseCost, cost);
          sigCostSum = __dadd_rn(sigCostSum, csig);
          if (lv) {
            sig = true;
            codedLevelAndDist = __dadd_rn(codedLevelAndDist, __dsub_rn(cost, csig));
            uncodedDist = __dadd_rn(uncodedDist, cost0);
          }
        }
        if (sig && (sb != shp.numSbb - 1 || anySigCG)) {
          double costZeroSB = baseCost;
          baseCost = __dadd_rn(baseCost, __dmul_rn(lambda, (double)bitsSigGroup[1]));
          costZeroSB = __dadd_rn(costZeroSB, __dmul_rn(lambda, (double)bitsSigGroup[0]));
          costZeroSB = __dadd_rn(costZeroSB, uncodedDist);
          costZeroSB = __dsub_rn(costZeroSB, codedLevelAndDist);
          costZeroSB = __dsub_rn(costZeroSB, sigCostSum);
          if (costZeroSB < baseCost) {
            sig = false;
            for (int i = 0; i < 16; i++) lvl[scn[sb * 16 + i] & 0xffffu] = 0;
          } else anySigCG = true;
        }
        if (sig) {
          sigGroups |= 1ull << sbPos;
          for (int i = 0; i < 16; i++) {
            const int blk = (int)(scn[sb * 16 + i] & 0xffffu);
            const int lv = lvl[blk];
            if (lv) {
              absSum += vabs(lv);
              level[blk] = lv;                         // the caller zero-filled the block
              const int qc = vmin(vmax(lv, inMin), inMax);
              int d;
              if (rightShift > 0) d = (qc * iScale + (1 << (rightShift - 1))) >> rightShift;
              else                d = (int)((unsigned)(qc * iScale) << (-rightShift));
              deq[blk] = vmin(vmax(d, -32768), 32767);
            }
          }
        }
      }
      P.results[ji].abs_sum_level = absSum;
    }
    __syncwarp();
  }
}

}  // namespace
