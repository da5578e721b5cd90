// vvc_intra_b200 -- RMD device kernels (sm_100a).  Included by vvcb_api.cu (the product) and, through a
// CUDA-on-pthreads shim, by tests/host_emul/emul_rmd.cpp (test-only lane emulation of this very source).
//
// Pipeline of one vvcb_rmd_eval call:
//   rmd_plan_count / rmd_plan_scan / rmd_plan_fill
//                      cut every visit into work items and bucket them: the eight small shapes (at most two lanes per slot) get one
//                      item per (visit, kind) in a bucket per (exact shape, kind); the larger shapes items of <= kItemTasks lane-tasks
//                      in a bucket per (SATD tile class of the shape) x (prediction kind: angular, planar/DC, MIP)
//   rmd_eval_kernel<TILE, KIND, MODE>   one launch per (tile class, kind) and item flavour (MODE 1: packed -- eight small visits per warp
//                      item; MODE 0: plain; MODE 2: plain + prediction samples out), dealt over several streams; persistent warps pull
//                      the bucket's items.  Every warp of a launch runs the same straight-line code (profiles/r1a: a monolithic kernel
//                      was instruction-fetch bound; profiles/r1z: so is any instantiation above ~45 KB).  A lane predicts one 8x8 (or
//                      4x4) unit of one evaluation slot, keeps the residual in registers, computes SAD and the Walsh-Hadamard SATD
//                      there, and the slot's lanes reduce with warp shuffles.
//   rmd_lists_kernel   one thread per visit: mode bits, double-precision costs and the exact replay of
//                      the reference's candidate-list insertions
#pragma once
#include "vvcb_core.cuh"

using namespace vvcb;

namespace {

#ifndef VVCB_EVAL_WARPS
#define VVCB_EVAL_WARPS 8
#endif
constexpr int kWarpsPerCta = VVCB_EVAL_WARPS;
constexpr int kThreads     = kWarpsPerCta * 32;
constexpr int KIND_ANG = 0, KIND_PDC = 1, KIND_MIP = 2;

// Reference lines and MIP inputs of one visit.  LMAX = kLineMax holds any CU; the packed kernels (several small visits per work
// item) use kLineSmall.
template <int LMAX> struct VisitSmem {
  int16_t lines[kNumSets][2][LMAX];       // [set][0 top / 1 left][index], tails replicated for positive angles
  int16_t mipBnd[8];                      // Haar-averaged boundary: [0..4) top, [4..8) left
  int16_t mipIn[2][8];                    // rebased MIP input vectors: [0] normal, [1] transposed orientation
  int     mipAux[4];                      // first boundary sample of each orientation, sum of each input vector
  int     pad;                            // odd number of words: the visits of a packed item start in different banks
};
using WarpSmem = VisitSmem<kLineMax>;

// ---- packed work items -------------------------------------------------------------------------------
// A visit of a small CU has few lane-tasks per prediction kind (8x8: 75 angular, 2-4 planar/DC, 19 MIP slots, one lane each), so a
// warp iteration that serves one visit runs mostly empty (profiles/r1z_summary.md: 22-26 of 32 lanes active in the angular kernels, 2-4 in the
// planar/DC ones).  Shapes of at most two lanes per slot are therefore planned into buckets of their own, one per exact shape, and
// the packed kernel instantiation takes kPackVisits visits of one shape at a time: their reference lines sit side by side in shared
// memory and the slots of all of them form one flat task list.
#ifndef VVCB_PACK_VISITS
#define VVCB_PACK_VISITS 8
#endif
constexpr int kPackVisits  = VVCB_PACK_VISITS;
constexpr int kLineSmall   = 52;          // sides <= 16: 2*16 + 1 + 3 + the replicated tail of 14 (16x4 on reference line 3)
constexpr int kSmallShapes = 8;
constexpr int kNumBucketsAll = kNumBuckets + kSmallShapes * kNumKinds;
static_assert((sizeof(VisitSmem<kLineSmall>) / 4) % 2 == 1, "bank stride of the packed line sets");

// index of the shape among the packed ones (4x4, 8x4, 4x8, 8x8, 16x4, 4x16, 16x8, 8x16), -1 for the larger shapes
__host__ __device__ __forceinline__ int small_shape_index(int lw, int lh)
{
  if (lw + lh > 7 || lw > 4 || lh > 4) return -1;
  if (lw == 2 && lh == 2) return 0;
  if (lw == 3 && lh == 2) return 1;
  if (lw == 2 && lh == 3) return 2;
  if (lw == 3 && lh == 3) return 3;
  if (lw == 4 && lh == 2) return 4;
  if (lw == 2 && lh == 4) return 5;
  if (lw == 4 && lh == 3) return 6;
  return 7;
}

struct PlanState {                        // device-resident, zeroed before every call
  unsigned count[kNumBucketsAll];         // items per bucket: [0, kNumBuckets) by (tile class, kind), then by (packed shape, kind)
  unsigned offset[kNumBucketsAll];        // first item of the bucket
  unsigned fill[kNumBucketsAll];          // fill cursor (plan) ...
  unsigned cursor[kNumBucketsAll];        // ... and consume cursor (eval)
};

// Position of (slot, visit) in the SAD / SATD scratch planes the evaluation kernels hand to the list kernel.  Visit-major: the ~100 values
// of a visit are written by one warp within a few microseconds into 448 contiguous bytes, so the partial-sector writes merge in L2 and most of the
// plane is still there when the list kernel reads it.  The slot-major layout of round 1 (coalesced for the list kernel, one thread per visit)
// scattered every store into a sector of its own: 2.10 GB of DRAM traffic per 1080p sweep against 0.68 GB now, list kernel 1.10 -> 1.02 ms
// (tools/scratch_layout_ab.sh, profiles/r2_summary.md).  VVCB_SCRATCH_VISIT_MAJOR=0 keeps the old layout for A/B builds.
#ifndef VVCB_SCRATCH_VISIT_MAJOR
#define VVCB_SCRATCH_VISIT_MAJOR 1
#endif
__host__ __device__ __forceinline__ size_t scratch_at(int slot, unsigned visit, int nVisits)
{
#if VVCB_SCRATCH_VISIT_MAJOR
  (void)nVisits;
  return (size_t)visit * VVCB_NUM_SLOTS + (size_t)slot;
#else
  return (size_t)slot * (size_t)nVisits + visit;
#endif
}

struct EvalParams {
  const vvcb_rmd_visit* visits;
  const WorkItem*       items;
  PlanState*            plan;
  uint32_t*             sadSM;    // scratch plane, indexed by scratch_at(slot, visit, nVisits)
  uint32_t*             satdSM;   // nullptr: only min(2 * SAD, SATD) is handed over, in sadSM (no detail tables were asked for: the lists need nothing else)
  int                   nVisits;
  const int16_t*        orig;
  const int16_t*        reco;
  int                   stride;   // both planes
  int                   bd, ctu;
  const Rom*            rom;
  int16_t*              predOut;  // optional: [slot][h][w] of visit 0 (debug / parity)
};

__device__ __forceinline__ bool visit_mrl_allowed(const vvcb_rmd_visit& v, int ctu)
{
  return !(v.flags & VVCB_VISIT_NO_MRL) && (v.y & (ctu - 1)) != 0;
}

__device__ __forceinline__ int visit_num_mip(const vvcb_rmd_visit& v)
{
  return (v.flags & VVCB_VISIT_NO_MIP) ? 0 : mip_num_modes(1 << v.log2w, 1 << v.log2h);
}

// position (1..5) of DC among MPM[1..5], 0 if absent: DC on reference lines 1/3 goes to the planar/DC kernel
__device__ __forceinline__ int mpm_dc_pos(const vvcb_rmd_visit& v)
{
  int pos = 0;
#pragma unroll
  for (int i = 5; i >= 1; i--) if (v.mpm[i] == 1) pos = i;
  return pos;
}

// slots of one kind for one visit
__device__ __forceinline__ int kind_slot_count(const vvcb_rmd_visit& v, int kind, int ctu)
{
  const bool mrl = visit_mrl_allowed(v, ctu);
  const int dc = mpm_dc_pos(v);
  if (kind == KIND_ANG) return 65 + (mrl ? 2 * (5 - (dc ? 1 : 0)) : 0);
  if (kind == KIND_PDC) return 2 + (mrl && dc ? 2 : 0);
  return visit_num_mip(v);
}

// index inside the kind's slot list -> evaluation slot (include/vvc_intra_b200.h)
__device__ __forceinline__ int kind_slot(const Rom& rom, const vvcb_rmd_visit& v, int kind, int idx)
{
  if (kind == KIND_MIP) return VVCB_SLOT_MIP + idx;
  const int dc = mpm_dc_pos(v);
  if (kind == KIND_PDC) {
    if (idx < 2) return idx;
    return (idx == 2 ? VVCB_SLOT_MRL1 : VVCB_SLOT_MRL3) + dc - 1;
  }
  if (idx < 65) return rom.angOrder[v.log2w - 2][v.log2h - 2][idx];
  const int per = 5 - (dc ? 1 : 0);
  const int j = idx - 65;
  const int li = j >= per ? 1 : 0;
  int i = 1 + (j - li * per);
  if (dc && i >= dc) i++;
  return (li ? VVCB_SLOT_MRL3 : VVCB_SLOT_MRL1) + i - 1;
}

// =====================================================================================================
// planning
// =====================================================================================================
__device__ __forceinline__ int items_of(int nSlots, int lanes, int& perItem, bool packed)
{
  if (packed) { perItem = nSlots; return nSlots ? 1 : 0; }     // a packed visit is one item per kind
  perItem = lanes >= kItemTasks ? 1 : kItemTasks / lanes;
  return (nSlots + perItem - 1) / perItem;
}

__device__ __forceinline__ int bucket_of(const Shape& sh, int kind, bool packed)
{
  const int small = packed ? small_shape_index(sh.lw, sh.lh) : -1;
  return small >= 0 ? kNumBuckets + small * kNumKinds + kind : sh.tile * kNumKinds + kind;
}

// Both planning passes aggregate per block in shared memory first: one global atomic per bucket per block.
__global__ void rmd_plan_count(const vvcb_rmd_visit* visits, int n, int ctu, PlanState* plan, int pack)
{
  __shared__ unsigned hist[kNumBucketsAll];
  if (threadIdx.x < kNumBucketsAll) hist[threadIdx.x] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const vvcb_rmd_visit v = visits[i];
    const Shape sh = make_shape(v.log2w, v.log2h);
    const bool packed = pack && small_shape_index(sh.lw, sh.lh) >= 0;
    for (int kind = 0; kind < kNumKinds; kind++) {
      int perItem;
      const int nItems = items_of(kind_slot_count(v, kind, ctu), sh.lanes, perItem, packed);
      if (nItems) atomicAdd(&hist[bucket_of(sh, kind, packed)], (unsigned)nItems);
    }
  }
  __syncthreads();
  if (threadIdx.x < kNumBucketsAll && hist[threadIdx.x]) atomicAdd(&plan->count[threadIdx.x], hist[threadIdx.x]);
}

__global__ void rmd_plan_scan(PlanState* plan)
{
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    unsigned acc = 0;
    for (int b = 0; b < kNumBucketsAll; b++) { plan->offset[b] = acc; acc += plan->count[b]; plan->fill[b] = 0; plan->cursor[b] = 0; }
  }
}

__global__ void rmd_plan_fill(const vvcb_rmd_visit* visits, int n, int ctu, PlanState* plan, WorkItem* items, int pack)
{
  __shared__ unsigned hist[kNumBucketsAll], base[kNumBucketsAll];
  if (threadIdx.x < kNumBucketsAll) hist[threadIdx.x] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  vvcb_rmd_visit v;
  Shape sh = make_shape(2, 2);
  unsigned local[kNumKinds] = { 0, 0, 0 };
  int nItems[kNumKinds] = { 0, 0, 0 }, perItem[kNumKinds] = { 1, 1, 1 }, nSlots[kNumKinds] = { 0, 0, 0 };
  bool packed = false;
  if (i < n) {
    v = visits[i];
    sh = make_shape(v.log2w, v.log2h);
    packed = pack && small_shape_index(sh.lw, sh.lh) >= 0;
    for (int kind = 0; kind < kNumKinds; kind++) {
      nSlots[kind] = kind_slot_count(v, kind, ctu);
      nItems[kind] = items_of(nSlots[kind], sh.lanes, perItem[kind], packed);
      if (nItems[kind]) local[kind] = atomicAdd(&hist[bucket_of(sh, kind, packed)], (unsigned)nItems[kind]);
    }
  }
  __syncthreads();
  if (threadIdx.x < kNumBucketsAll && hist[threadIdx.x])
    base[threadIdx.x] = plan->offset[threadIdx.x] + atomicAdd(&plan->fill[threadIdx.x], hist[threadIdx.x]);
  __syncthreads();
  if (i < n)
    for (int kind = 0; kind < kNumKinds; kind++) {
      const unsigned at = base[bucket_of(sh, kind, packed)] + local[kind];
      for (int k = 0; k < nItems[kind]; k++) {
        WorkItem w;
        w.visit = (uint32_t)i;
        w.slot_begin = (uint16_t)(k * perItem[kind]);
        w.slot_count = (uint16_t)vmin(perItem[kind], nSlots[kind] - k * perItem[kind]);
        items[at + k] = w;
      }
    }
}

// The three planning passes in one launch of one CTA, for the walk-sized batches of vvcb_cu_eval (a few dozen visits; plan state need not be
// zeroed beforehand).  The order of the items inside a bucket differs from the three-kernel plan; nothing depends on it.
__global__ void __launch_bounds__(256) rmd_plan_small(const vvcb_rmd_visit* visits, int n, int ctu, PlanState* plan, WorkItem* items, int pack)
{
  __shared__ unsigned cnt[kNumBucketsAll], off[kNumBucketsAll], cur[kNumBucketsAll];
  for (int b = threadIdx.x; b < kNumBucketsAll; b += blockDim.x) cnt[b] = 0;
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const vvcb_rmd_visit v = visits[i];
    const Shape sh = make_shape(v.log2w, v.log2h);
    const bool packed = pack && small_shape_index(sh.lw, sh.lh) >= 0;
    for (int kind = 0; kind < kNumKinds; kind++) {
      int perItem;
      const int nItems = items_of(kind_slot_count(v, kind, ctu), sh.lanes, perItem, packed);
      if (nItems) atomicAdd(&cnt[bucket_of(sh, kind, packed)], (unsigned)nItems);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned acc = 0;
    for (int b = 0; b < kNumBucketsAll; b++) {
      off[b] = acc; cur[b] = 0;
      plan->count[b] = cnt[b]; plan->offset[b] = acc; plan->fill[b] = cnt[b]; plan->cursor[b] = 0;
      acc += cnt[b];
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const vvcb_rmd_visit v = visits[i];
    const Shape sh = make_shape(v.log2w, v.log2h);
    const bool packed = pack && small_shape_index(sh.lw, sh.lh) >= 0;
    for (int kind = 0; kind < kNumKinds; kind++) {
      int perItem;
      const int nSlots = kind_slot_count(v, kind, ctu);
      const int nItems = items_of(nSlots, sh.lanes, perItem, packed);
      if (!nItems) continue;
      const int b = bucket_of(sh, kind, packed);
      const unsigned at = off[b] + atomicAdd(&cur[b], (unsigned)nItems);
      for (int k = 0; k < nItems; k++) {
        WorkItem w;
        w.visit = (uint32_t)i;
        w.slot_begin = (uint16_t)(k * perItem);
        w.slot_count = (uint16_t)vmin(perItem, nSlots - k * perItem);
        items[at + k] = w;
      }
    }
  }
}

// =====================================================================================================
// reference lines of one visit into the warp's shared memory
// =====================================================================================================
// One entry of a line set: walk position i (past the walk: the replicated tails) -> the sample, or mid-grey when nothing is available.
// The load is issued here; the caller stores it with store_line_entry once all the loads of its batch are in flight.
struct LineCtx { LineGeom g; int extTop, extLeft, nTop, nLeft, total; };

template <int UNIT = 4> __device__ __forceinline__ LineCtx make_line_ctx(const vvcb_rmd_visit& v, const Shape& sh, int mrl)
{
  LineCtx c;
  c.g = make_line_geom<UNIT>(v, sh.w, sh.h, mrl);
  // tails: the main reference of positive angles is extended by replication (CL/IntraPrediction.cpp:717-726)
  c.extTop = (mrl << vmax(0, sh.lw - sh.lh)) + 2; c.extLeft = (mrl << vmax(0, sh.lh - sh.lw)) + 2;
  c.nTop = 2 * sh.w + 1 + mrl; c.nLeft = 2 * sh.h + 1 + mrl;
  c.total = c.g.n + c.extTop + c.extLeft;
  return c;
}

__device__ __forceinline__ int load_line_entry(const LineCtx& c, const int16_t* base, int stride, int bd, int i)
{
  const int pos = i < c.g.n ? i : (i < c.g.n + c.extTop ? c.g.n - 1 : 0);
  const int src = line_source(c.g, pos);
  int val = 1 << (bd - 1);
  if (src >= 0) {
    bool isLeft; int k, dx, dy;
    line_pos(c.g, src, isLeft, k, dx, dy);
    val = base[dy * stride + dx];
  }
  return val;
}

#if defined(__CUDACC__)
#define VVCB_EMUL_ASSERT(x)
#else
#include <assert.h>
#define VVCB_EMUL_ASSERT(x) assert(x)          // host emulation of this source (tests/host_emul): bounds of the shared-memory lines
#endif

template <class SM>
__device__ __forceinline__ void store_line_entry(SM& sm, int set, const LineCtx& c, int i, int val)
{
  VVCB_EMUL_ASSERT(c.nTop + c.extTop <= (int)(sizeof(sm.lines[0][0]) / sizeof(int16_t)) && c.nLeft + c.extLeft <= (int)(sizeof(sm.lines[0][0]) / sizeof(int16_t)));
  if (i < c.g.n) {
    bool isLeft; int k, dx, dy;
    line_pos(c.g, i, isLeft, k, dx, dy);
    if (isLeft) sm.lines[set][1][k] = (int16_t)val;
    else {
      sm.lines[set][0][k] = (int16_t)val;
      if (k == 0) sm.lines[set][1][0] = (int16_t)val;
    }
  } else if (i < c.g.n + c.extTop) sm.lines[set][0][c.nTop + (i - c.g.n)] = (int16_t)val;
  else sm.lines[set][1][c.nLeft + (i - c.g.n - c.extTop)] = (int16_t)val;
}

// Reference line 0 (set 0) of one visit, or -- NS == 3 -- lines 0, 1 and 3 (sets 0, 2, 3), straight from the reconstruction plane.
// Every lane issues the loads of two walk positions of all NS lines before it stores any of them, so a small CU costs one memory
// round trip instead of one per line and 32 positions -- at the price of 2 NS inlined copies of the walk arithmetic.
template <int NS, class SM>
__device__ void build_line_sets(SM& sm, const vvcb_rmd_visit& v, const Shape& sh, const int16_t* reco, int stride, int bd, int lane)
{
  const int16_t* base = reco + (size_t)v.y * stride + v.x;
  LineCtx c[NS];
#pragma unroll
  for (int q = 0; q < NS; q++) c[q] = make_line_ctx(v, sh, q == 2 ? 3 : q);
  const int total = c[NS - 1].total;               // the longest walk
#pragma unroll 1
  for (int i0 = lane; i0 < total; i0 += 64) {
    int val[NS][2];
#pragma unroll
    for (int q = 0; q < NS; q++)
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int i = i0 + 32 * u;
        val[q][u] = i < c[q].total ? load_line_entry(c[q], base, stride, bd, i) : 0;
      }
#pragma unroll
    for (int q = 0; q < NS; q++)
#pragma unroll
      for (int u = 0; u < 2; u++) {
        const int i = i0 + 32 * u;
        if (i < c[q].total) store_line_entry(sm, q ? q + 1 : 0, c[q], i, val[q][u]);
      }
  }
}

// one line set (TU prediction kernel: a job needs line 0 and at most one more); UNIT as make_line_geom
template <int UNIT = 4, class SM>
__device__ void build_line_set(SM& sm, int set, int mrl, const vvcb_rmd_visit& v, const Shape& sh,
                               const int16_t* reco, int stride, int bd, int lane)
{
  const LineCtx c = make_line_ctx<UNIT>(v, sh, mrl);
  const int16_t* base = reco + (size_t)v.y * stride + v.x;
  for (int i = lane; i < c.total; i += 32) store_line_entry(sm, set, c, i, load_line_entry(c, base, stride, bd, i));
}

// [1 2 1]/4 smoothing of set 0 into set 1 (CL/IntraPrediction.cpp:1470-1522), tails copied
template <class SM>
__device__ void build_filtered_set(SM& sm, const Shape& sh, int lane)
{
  const int nTop = 2 * sh.w + 1, nLeft = 2 * sh.h + 1;
  const int16_t* top = sm.lines[0][0];
  const int16_t* left = sm.lines[0][1];
  for (int i = lane; i < nTop + 2; i += 32) {
    int v;
    if (i == 0) v = (left[1] + 2 * top[0] + top[1] + 2) >> 2;
    else if (i >= nTop - 1) v = top[i];
    else v = (top[i - 1] + 2 * top[i] + top[i + 1] + 2) >> 2;
    sm.lines[1][0][i] = (int16_t)v;
    if (i == 0) sm.lines[1][1][0] = (int16_t)v;
  }
  for (int i = 1 + lane; i < nLeft + 2; i += 32) {
    int v;
    if (i >= nLeft - 1) v = left[i];
    else v = (left[i - 1] + 2 * left[i] + left[i + 1] + 2) >> 2;   // left[0] == top[0]
    sm.lines[1][1][i] = (int16_t)v;
  }
}

// MIP inputs of one visit (CL/MatrixIntraPrediction.cpp:71-124): Haar-averaged boundary, then the two rebased
// input vectors (normal and transposed orientation) with their sums.
template <class SM>
__device__ void build_mip_inputs(SM& sm, const Shape& sh, const MipGeom& mg, int bd, int lane)
{
  if (lane < 8) {
    const int side = lane >> 2, i = lane & 3;          // 0 top, 1 left
    if (i < mg.bsz) {
      const int len = side ? sh.h : sh.w;
      const int f = len / mg.bsz;
      const int16_t* src = sm.lines[0][side] + 1 + i * f;
      int s = 0;
      for (int k = 0; k < f; k++) s += src[k];
      sm.mipBnd[side * 4 + i] = (int16_t)(f == 1 ? s : (s + (f >> 1)) >> vlog2(f));
    }
  }
  __syncwarp();
  if (lane < 16) {
    const int t = lane >> 3, i = lane & 7;
    const int first = sm.mipBnd[t ? 4 : 0];
    int val = 0;
    if (i < 2 * mg.bsz) {
      const int raw = i < mg.bsz ? sm.mipBnd[(t ? 4 : 0) + i] : sm.mipBnd[(t ? 0 : 4) + i - mg.bsz];
      val = i == 0 ? (mg.small ? first - (1 << (bd - 1)) : 0) : raw - first;
    }
    sm.mipIn[t][i] = (int16_t)val;
    if (i == 0) sm.mipAux[t] = first;
  }
  __syncwarp();
  if (lane < 2) {
    int sum = 0;
    for (int i = 0; i < 8; i++) sum += sm.mipIn[lane][i];
    sm.mipAux[2 + lane] = sum;
  }
}

// =====================================================================================================
// per-slot pieces
// =====================================================================================================
__device__ __forceinline__ SlotInfo make_slot_info(const Rom& rom, const vvcb_rmd_visit& v, const Shape& sh, int slot)
{
  SlotInfo s;
  s.mrl = 0; s.set = 0;
  if (slot >= VVCB_SLOT_MIP) { s.kind = 3; s.mode = slot - VVCB_SLOT_MIP; s.p = ModeParam{}; return s; }
  if (slot >= VVCB_SLOT_MRL1) {
    const int li = slot >= VVCB_SLOT_MRL3 ? 1 : 0;
    s.mrl  = li ? 3 : 1;
    s.set  = 2 + li;
    s.mode = v.mpm[1 + (slot - VVCB_SLOT_MRL1) % 5];
    s.p    = rom.mode[sh.lw - 2][sh.lh - 2][s.mode];
    s.p.ref_filter = 0; s.p.interp = 0; s.p.pdpc = 0;      // CL/IntraPrediction.cpp:509, :559-575
  } else {
    s.mode = slot;
    s.p    = rom.mode[sh.lw - 2][sh.lh - 2][slot];
    s.set  = s.p.ref_filter ? 1 : 0;
  }
  s.kind = s.mode == 0 ? 0 : (s.mode == 1 ? 1 : 2);
  return s;
}

// Main reference of a negative-angle slot with its projected extension (CL/IntraPrediction.cpp:654-673):
// buf[t + mh] = refMain0[t], t in [-mh, mw + 1 + mrl].  Positive angles read the visit's lines directly.
template <class SM>
__device__ void build_projected_line(int16_t* buf, const SM& sm, const SlotInfo& s, int mw, int mh, int gl, int gsize)
{
  const int16_t* mainSrc = sm.lines[s.set][s.p.is_ver ? 0 : 1];
  const int16_t* sideSrc = sm.lines[s.set][s.p.is_ver ? 1 : 0];
  const int inv = s.p.inv_angle;
  // projected part, t in [-mh, -1]
  for (int i = gl; i < mh; i += gsize) buf[i] = sideSrc[vmin(((mh - i) * inv + 256) >> 9, mh)];
  // straight part, t in [0, mw + 1 + mrl], two samples per move: mh is even, the line arrays and the slot scratch are word aligned
  // (an odd count copies one sample past the end: inside both arrays, never read)
  const uint32_t* src2 = reinterpret_cast<const uint32_t*>(mainSrc);
  uint32_t* dst2 = reinterpret_cast<uint32_t*>(buf + mh);
  const int words = (mw + 3 + s.mrl) >> 1;
  for (int i = gl; i < words; i += gsize) dst2[i] = src2[i];
}

// residual of one R x C piece against the original block, SAD accumulated.  TRANSPOSED: the prediction q is in the
// main/side frame of a horizontal mode, i.e. q[i][j] predicts block sample (y0 + j, x0 + i); SAD and the sum of
// absolute Hadamard coefficients are invariant under transposition, so the residual stays in that frame.
// org points at block sample (y0, x0) of the piece.
template <int R, int C, bool TRANSPOSED>
__device__ __forceinline__ void residual_unit(const int16_t* org, int stride, const int (&q)[R][C], int (&d)[R][C], int& sad)
{
  constexpr int ROWS = TRANSPOSED ? C : R, COLS = TRANSPOSED ? R : C;   // extent of the piece in the picture
#pragma unroll
  for (int r = 0; r < ROWS; r++) {
    const int16_t* row = org + r * stride;
#pragma unroll
    for (int c = 0; c < COLS; c += 4) {
      const uint2 v = *reinterpret_cast<const uint2*>(row + c);       // CU positions are multiples of 4 samples
      const int o0 = (int)(int16_t)(v.x & 0xffff), o1 = (int)(int16_t)(v.x >> 16);
      const int o2 = (int)(int16_t)(v.y & 0xffff), o3 = (int)(int16_t)(v.y >> 16);
      if (TRANSPOSED) {
        d[c + 0][r] = o0 - q[c + 0][r]; d[c + 1][r] = o1 - q[c + 1][r];
        d[c + 2][r] = o2 - q[c + 2][r]; d[c + 3][r] = o3 - q[c + 3][r];
        sad = vsad(o0, q[c + 0][r], sad); sad = vsad(o1, q[c + 1][r], sad);
        sad = vsad(o2, q[c + 2][r], sad); sad = vsad(o3, q[c + 3][r], sad);
      } else {
        d[r][c + 0] = o0 - q[r][c + 0]; d[r][c + 1] = o1 - q[r][c + 1];
        d[r][c + 2] = o2 - q[r][c + 2]; d[r][c + 3] = o3 - q[r][c + 3];
        sad = vsad(o0, q[r][c + 0], sad); sad = vsad(o1, q[r][c + 1], sad);
        sad = vsad(o2, q[r][c + 2], sad); sad = vsad(o3, q[r][c + 3], sad);
      }
    }
  }
}

// q[i][j] is block sample (y0 + i, x0 + j), or (y0 + j, x0 + i) when transposed
template <int R, int C>
__device__ __forceinline__ void store_pred(int16_t* out, int w, int x0, int y0, bool transposed, const int (&q)[R][C])
{
#pragma unroll
  for (int i = 0; i < R; i++)
#pragma unroll
    for (int j = 0; j < C; j++) {
      if (transposed) out[(y0 + j) * w + x0 + i] = (int16_t)q[i][j];
      else            out[(y0 + i) * w + x0 + j] = (int16_t)q[i][j];
    }
}

// =====================================================================================================
// prediction of one unit per kind.  q is produced in the frame named by `transposed`.
// =====================================================================================================
// (x0, y0): block position of the lane's unit; rOff: first row of the piece inside the unit, counted along the side
// direction of the prediction frame (block rows for vertical modes, block columns for horizontal ones)
template <int R, int C, class SM>
__device__ __forceinline__ void predict_angular(const SM& sm, const int16_t* projected, const SlotInfo& s, const Shape& sh,
                                                const uint32_t* filt, int bd, int x0, int y0, int rOff, int (&q)[R][C])
{
  const bool ver = s.p.is_ver;
  const int mw = ver ? sh.w : sh.h, mh = ver ? sh.h : sh.w;
  const int16_t* ml = s.p.angle < 0 ? projected + mh : sm.lines[s.set][ver ? 0 : 1];
  pred_angular_unit<R, C>(ml, sm.lines[s.set][ver ? 1 : 0], s.p, s.mrl, mw, mh, ver ? x0 : y0, (ver ? y0 : x0) + rOff, filt, (1 << bd) - 1, q);
}

// MIP: first interpolation pass of one slot into shared memory (CL/MatrixIntraPrediction.cpp:469-567,
// shorter side first).  w >= h: plane[y * redW + rx] (vertical pass at the reduced columns);
// h > w: plane[ry * w + x] (horizontal pass at the reduced rows).
// When that first pass is the identity (no up-sampling along the shorter side) the plane IS the reduced prediction.
__device__ __forceinline__ int mip_plane_offset(const MipGeom& mg, const Shape& sh)
{
  const bool identity = sh.h > sh.w ? mg.upH == 1 : mg.upV == 1;
  return identity ? 0 : mg.redW * mg.redH;
}

template <class SM>
__device__ void build_mip_planes(int16_t* red, int16_t* plane, const Rom& rom, const SM& sm, const MipGeom& mg, const Shape& sh,
                                 int bd, int mode, int gl, int gsize)
{
  const MipSlot ms = make_mip_slot(rom.mip + mip_family_base(mg.family), mg, sm.mipIn, sm.mipAux, mode);
  const int nRed = mg.redW * mg.redH, maxv = (1 << bd) - 1;
  for (int i = gl; i < nRed; i += gsize)
    red[i] = (int16_t)mip_reduced_sample(ms, mg, sh.w, sh.h, maxv, i & (mg.redW - 1), i >> mg.lgRedW);
  __syncwarp();
  if (plane == red) return;
  const int16_t* top = sm.lines[0][0];
  const int16_t* left = sm.lines[0][1];
  if (sh.h > sh.w) {
    const int n = mg.redH << sh.lw;
    for (int i = gl; i < n; i += gsize) {
      const int ry = i >> sh.lw, x = i & (sh.w - 1);
      const int rx = x >> mg.lgUpH, k = (x & (mg.upH - 1)) + 1;
      const int row = mg.upV * (ry + 1) - 1;
      const int before = rx == 0 ? left[1 + row] : red[(ry << mg.lgRedW) + rx - 1];
      const int behind = red[(ry << mg.lgRedW) + rx];
      plane[i] = (int16_t)(((mg.upH - k) * before + k * behind + (mg.upH >> 1)) >> mg.lgUpH);
    }
  } else {
    const int n = sh.h << mg.lgRedW;
    for (int i = gl; i < n; i += gsize) {
      const int y = i >> mg.lgRedW, rx = i & (mg.redW - 1);
      const int ry = y >> mg.lgUpV, k = (y & (mg.upV - 1)) + 1;
      const int col = mg.upH * (rx + 1) - 1;
      const int before = ry == 0 ? top[1 + col] : red[((ry - 1) << mg.lgRedW) + rx];
      const int behind = red[(ry << mg.lgRedW) + rx];
      plane[i] = (int16_t)(((mg.upV - k) * before + k * behind + (mg.upV >> 1)) >> mg.lgUpV);
    }
  }
}

template <int R, int C, class SM>
__device__ __forceinline__ void predict_mip(const SM& sm, const int16_t* plane, const MipGeom& mg, const Shape& sh,
                                            int x0, int y0, int (&q)[R][C])
{
  const int16_t* top = sm.lines[0][0];
  const int16_t* left = sm.lines[0][1];
  if (sh.h > sh.w) {
    // second pass vertical; plane[ry * w + x] holds the rows that carry reduced samples
#pragma unroll
    for (int i = 0; i < R; i++) {
      const int y = y0 + i;
      const int ry = y >> mg.lgUpV, k = (y & (mg.upV - 1)) + 1;
      const int16_t* rowB = plane + (ry << sh.lw) + x0;
#pragma unroll
      for (int j = 0; j < C; j++) {
        const int before = ry == 0 ? top[1 + x0 + j] : rowB[j - sh.w];
        q[i][j] = ((mg.upV - k) * before + k * rowB[j] + (mg.upV >> 1)) >> mg.lgUpV;
      }
    }
  } else {
    // second pass horizontal; plane[y * redW + rx] holds the columns that carry reduced samples
#pragma unroll
    for (int i = 0; i < R; i++) {
      const int y = y0 + i;
      const int16_t* rowP = plane + (y << mg.lgRedW);
#pragma unroll
      for (int j = 0; j < C; j++) {
        const int x = x0 + j;
        const int rx = x >> mg.lgUpH, k = (x & (mg.upH - 1)) + 1;
        const int before = rx == 0 ? left[1 + y] : rowP[rx - 1];
        q[i][j] = ((mg.upH - k) * before + k * rowP[rx] + (mg.upH >> 1)) >> mg.lgUpH;
      }
    }
  }
}

// MIP prediction of piece k of a slot that one lane owns: the packed 4x4, 8x4, 4x8 and 8x8 shapes, one per tile class TILE 0..3
// (4x4 matrices for 4x4, 8x8 matrices for the others; a 4 x 4 reduced block).  The reduced samples the piece needs are computed in
// registers and up-sampled there (CL/MatrixIntraPrediction.cpp:469-567), with no plane in shared memory and no pass for an identity
// direction.  Pieces come in order k = 0, 1 (4x4: k = 0 only): 8x4 takes reduced columns 2k, 2k + 1, 4x8 and 8x8 reduced rows 2k, 2k + 1;
// `carry` hands piece 1 the last reduced column / row of piece 0, the sample before its first one.
template <int TILE, int R, int C, class SM>
__device__ __forceinline__ void predict_mip_lane(const SM& sm, const MipSlot& ms, int k, int maxv, int (&carry)[4], int (&q)[R][C])
{
  const int16_t* top = sm.lines[0][0];
  const int16_t* left = sm.lines[0][1];
  // matrix row of reduced sample (ry, rx): ry * 4 + rx, transposed modes rx * 4 + ry
  const int stepY = ms.transpose ? 1 : 4, stepX = ms.transpose ? 4 : 1;
  if constexpr (TILE == 0) {
#pragma unroll
    for (int i = 0; i < 4; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) q[i][j] = mip_row_sample<false>(ms, i * stepY + j * stepX, maxv);
  } else if constexpr (TILE == 1) {
    // 8x4: the vertical pass is the identity; horizontal up-sampling by 2 from the left boundary
#pragma unroll
    for (int i = 0; i < 4; i++) {
      const int b  = k ? carry[i] : left[1 + i];
      const int r0 = mip_row_sample<true>(ms, i * stepY + 2 * k * stepX, maxv);
      const int r1 = mip_row_sample<true>(ms, i * stepY + (2 * k + 1) * stepX, maxv);
      q[i][0] = (b + r0 + 1) >> 1; q[i][1] = r0; q[i][2] = (r0 + r1 + 1) >> 1; q[i][3] = r1;
      carry[i] = r1;
    }
  } else {
    // 4x8, 8x8: vertical up-sampling by 2 from the top boundary (at the reduced columns), then for 8x8 horizontal by 2 from the left one
    int v[4][4];
#pragma unroll
    for (int rx = 0; rx < 4; rx++) {
      const int b  = k ? carry[rx] : top[TILE == 3 ? 2 + 2 * rx : 1 + rx];
      const int r0 = mip_row_sample<true>(ms, 2 * k * stepY + rx * stepX, maxv);
      const int r1 = mip_row_sample<true>(ms, (2 * k + 1) * stepY + rx * stepX, maxv);
      v[0][rx] = (b + r0 + 1) >> 1; v[1][rx] = r0; v[2][rx] = (r0 + r1 + 1) >> 1; v[3][rx] = r1;
      carry[rx] = r1;
    }
    if constexpr (TILE == 2) {
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) q[i][j] = v[i][j];
    } else {
#pragma unroll
      for (int i = 0; i < 4; i++) {
        const int l = left[1 + 4 * k + i];
#pragma unroll
        for (int rx = 0; rx < 4; rx++) {
          q[i][2 * rx]     = ((rx ? v[i][rx - 1] : l) + v[i][rx] + 1) >> 1;
          q[i][2 * rx + 1] = v[i][rx];
        }
      }
    }
  }
}

// =====================================================================================================
// the evaluation kernel, one instantiation per (SATD tile class, prediction kind)
// =====================================================================================================
#ifndef VVCB_EVAL_MIN_CTAS
#define VVCB_EVAL_MIN_CTAS 2
#endif
// PACK = false: one work item = a slot range of one visit (any shape).  PACK = true: one work item = up to kPackVisits visits of one
// small shape with all their slots of this kind; half as many warps per CTA (their shared memory holds kPackVisits line sets each).
template <bool PACK> struct EvalCfg {
  static constexpr int kWarps   = PACK ? kWarpsPerCta / 2 : kWarpsPerCta;
  static constexpr int kThreads = kWarps * 32;
  static constexpr int kMinCtas = PACK ? 2 * VVCB_EVAL_MIN_CTAS : VVCB_EVAL_MIN_CTAS;
  static constexpr int kVisits  = PACK ? kPackVisits : 1;
  using Smem = VisitSmem<PACK ? kLineSmall : kLineMax>;
};

// the packed shapes of a tile class, in bucket order
__host__ __device__ __forceinline__ int pack_shape_count(int tile) { return tile == 1 || tile == 2 ? 2 : 1; }
__host__ __device__ __forceinline__ int pack_shape(int tile, int i)
{
  return tile == 0 ? 0 : tile == 1 ? (i ? 4 : 1) : tile == 2 ? (i ? 5 : 2) : tile == 3 ? 3 : tile == 4 ? 6 : 7;
}

// MODE 0: plain items; MODE 1: packed items; MODE 2: plain items + the prediction samples of visit 0 written to P.predOut (the parity /
// integration entry points vvcb_rmd_pred*; kept out of the throughput kernels: 350 instructions in the middle of their hot loop)
// The shared memory of one evaluation CTA, as one block: the per-bucket kernels declare it statically, the any-bucket kernels (below) hand
// the same layout to whichever bucket their CTA serves.
template <bool PACK> struct EvalShared {
  using Cfg = EvalCfg<PACK>;
  typename Cfg::Smem smem[Cfg::kWarps][Cfg::kVisits];
  int16_t sScratch[Cfg::kWarps][kSlotLineWords];                  // per-slot scratch of the slots in flight
  vvcb_rmd_visit sVisit[Cfg::kWarps][Cfg::kVisits];
  int sSlots[Cfg::kWarps][Cfg::kVisits + 1];                      // packed items: number of slots of each visit
  unsigned sIndex[Cfg::kWarps][Cfg::kVisits];                     // the visits' indices in the batch
  uint32_t sFilt[64];
};

// MIP slots that one lane owns (4x4, 8x4, 4x8, 8x8) are predicted in registers (predict_mip_lane), with the matrices of their family
// (4x4 for the 4x4 class, 8x8 for the others) copied to shared memory: at most 1 360 bytes, which fit under the 48 KB of static shared
// memory beside EvalShared; the slots of larger shapes read theirs from the ROM in global memory.  The lane-owned shapes come in packed
// items, and in plain items only for the prediction-output kernels (MODE 2).
template <int TILE, int KIND, int MODE> constexpr bool kLaneMip = KIND == KIND_MIP && TILE < 4 && MODE != 0;
constexpr int kMipLaneWords = 10 * 34;       // the larger of mip_family_words(0), mip_family_words(1)

// sMip: kMipLaneWords of shared memory when kLaneMip<TILE, KIND, MODE>
template <int TILE, int KIND, int MODE>
__device__ __forceinline__ void rmd_eval_body(const EvalParams& P, EvalShared<MODE == 1>& shm, uint32_t* sMip)
{
  constexpr bool PACK = MODE == 1, WITH_PRED = MODE == 2;
  using Cfg = EvalCfg<PACK>;
  using SM = typename Cfg::Smem;
  constexpr int S = TILE < 3 ? 4 : 8;
  constexpr int V = Cfg::kVisits;
  constexpr bool LANE_MIP = kLaneMip<TILE, KIND, MODE>;
  constexpr bool ONLY_LANE_MIP = LANE_MIP && PACK && (TILE == 0 || TILE == 3);    // the packed 4x4 and 8x8 classes hold nothing else
  constexpr int MIP_FAMILY = TILE == 0 ? 0 : 1;
  auto& smem = shm.smem;
  auto& sScratch = shm.sScratch;
  auto& sVisit = shm.sVisit;
  auto& sSlots = shm.sSlots;
  auto& sIndex = shm.sIndex;
  auto& sFilt = shm.sFilt;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x < 64) sFilt[threadIdx.x] = (&P.rom->filt[0][0])[threadIdx.x];
  if (LANE_MIP)
    for (int i = threadIdx.x; i < mip_family_words(MIP_FAMILY); i += Cfg::kThreads) sMip[i] = P.rom->mip[mip_family_base(MIP_FAMILY) + i];
  __syncthreads();
  const Rom& rom = *P.rom;

#pragma unroll 1
  for (int ps = 0; ps < (PACK ? pack_shape_count(TILE) : 1); ps++) {
  const int BUCKET = PACK ? kNumBuckets + pack_shape(TILE, ps) * kNumKinds + KIND : TILE * kNumKinds + KIND;
  const unsigned nItems = P.plan->count[BUCKET];
  const WorkItem* items = P.items + P.plan->offset[BUCKET];

  for (;;) {
    unsigned it = 0;
    if (lane == 0) it = atomicAdd(&P.plan->cursor[BUCKET], (unsigned)V);
    it = __shfl_sync(0xffffffffu, it, 0);
    if (it >= nItems) break;
    const int nv = PACK ? (int)(nItems - it < (unsigned)V ? nItems - it : (unsigned)V) : 1;
    const WorkItem item = items[it];                  // PACK: slot range = all slots of the kind, for every visit of the item
    __syncwarp();
    // ---- the item's visits into shared memory (20 words each)
#pragma unroll 1
    for (int i = lane; i < nv * 20; i += 32) {
      const int j = i / 20, k = i - j * 20;
      reinterpret_cast<uint32_t*>(&sVisit[warp][j])[k] = reinterpret_cast<const uint32_t*>(P.visits + items[it + j].visit)[k];
    }
    if (lane < nv) sIndex[warp][lane] = items[it + lane].visit;
    __syncwarp();
    const Shape sh = make_shape(sVisit[warp][0].log2w, sVisit[warp][0].log2h);    // one shape per packed item
    const MipGeom mg = make_mip_geom(sh.w, sh.h);
    // Task list of a packed item, slot-major: task = ((slot index * V + visit) * lanes + unit), so that the 32 lanes of a warp
    // iteration work on the same few slot indices of all the visits -- the angular slots are ordered by (hor / ver, PDPC class)
    // per shape, which keeps projection, PDPC and transposition branches uniform across the iteration (profiles/r1z_summary.md: with the
    // visits' slots laid end to end 21.5 of 32 lanes were active per instruction).
    int maxSlots = PACK ? 0 : (int)item.slot_count;
    if (PACK) {
      int c = lane < nv ? kind_slot_count(sVisit[warp][lane], KIND, P.ctu) : 0;
      if (lane < V) sSlots[warp][lane] = c;
      for (int o = V >> 1; o > 0; o >>= 1) c = vmax(c, __shfl_xor_sync(0xffffffffu, c, o));
      maxSlots = __shfl_sync(0xffffffffu, c, 0);
    }

    // ---- reference lines needed by the item's slots (loops kept rolled: code size, profiles/r1z_summary.md)
#pragma unroll 1
    for (int j = 0; j < nv; j++) {
      const vvcb_rmd_visit& v = sVisit[warp][j];
      SM& sm = smem[warp][j];
      int nSets = 1;                             // line 0, plus lines 1 and 3 when the item holds MRL slots (they end the kind's list)
      if (KIND != KIND_MIP) {
        const int lastSlot = kind_slot(rom, v, KIND, PACK ? kind_slot_count(v, KIND, P.ctu) - 1 : item.slot_begin + item.slot_count - 1);
        if (lastSlot >= VVCB_SLOT_MRL1) nSets = 3;
      }
      if (KIND == KIND_PDC) {
        // planar / DC items are all set-up (one warp iteration of arithmetic): overlap the loads of the lines
        if (nSets == 3) build_line_sets<3>(sm, v, sh, P.reco, P.stride, P.bd, lane);
        else            build_line_sets<1>(sm, v, sh, P.reco, P.stride, P.bd, lane);
      } else {
        // angular / MIP kernels: one rolled copy (their hot loops feel every extra KB of code, profiles/r1z_summary.md)
#pragma unroll 1
        for (int q = 0; q < nSets; q++) build_line_set(sm, q ? q + 1 : 0, q == 2 ? 3 : q, v, sh, P.reco, P.stride, P.bd, lane);
      }
    }
    __syncwarp();
#pragma unroll 1
    for (int j = 0; j < nv; j++) {
      if (KIND != KIND_MIP) build_filtered_set(smem[warp][j], sh, lane);
      else                  build_mip_inputs(smem[warp][j], sh, mg, P.bd, lane);
    }
    __syncwarp();

    const int lanes = sh.lanes;                       // lanes per slot
    const int gsize = lanes > 32 ? 32 : lanes;        // lanes of one slot inside this warp iteration
    const int lgG   = lanes > 32 ? 5 : sh.lgLanes;
    const int gidx  = lane >> lgG, gl = lane & (gsize - 1);
    int16_t* scratch = sScratch[warp] + gidx * ((kSlotLineWords / 32) << lgG);
    // visits interleaved in the task list: V, or the next power of two when the item holds fewer (the tail of a bucket; single-visit calls)
    const int lgV = !PACK ? 0 : nv > 4 ? 3 : nv > 2 ? 2 : nv > 1 ? 1 : 0;
    const int nTasks = (maxSlots << lgV) * lanes;
    int accSad = 0, accSatd = 0;

    for (int base = 0; base < nTasks; base += 32) {
      const int task = base + lane;
      bool act = task < nTasks;
      int tk = act ? task : nTasks - 1;
      int vi = 0;
      if (PACK) {
        const int r = tk >> sh.lgLanes;
        vi = r & ((1 << lgV) - 1);
        int idx = r >> lgV;
        act = act && vi < nv && idx < sSlots[warp][vi];
        if (vi >= nv) vi = nv - 1;                                   // idle lanes shadow a real task
        if (idx >= sSlots[warp][vi]) idx = sSlots[warp][vi] - 1;
        tk = (idx << sh.lgLanes) | (tk & (lanes - 1));
      }
      const vvcb_rmd_visit& v = sVisit[warp][vi];
      const SM& sm = smem[warp][vi];
      const unsigned vIdx = sIndex[warp][vi];
      const int16_t* org = P.orig + (size_t)v.y * P.stride + v.x;
      const int u = tk & (lanes - 1);
      const int slot = kind_slot(rom, v, KIND, (PACK ? 0 : item.slot_begin) + (tk >> sh.lgLanes));
      const SlotInfo s = make_slot_info(rom, v, sh, slot);

      // ---- per-slot scratch built by the slot's lanes
      __syncwarp();
      int dc = 0;
      const bool laneMip = ONLY_LANE_MIP || (LANE_MIP && lanes == 1);     // uniform over the warp: one shape per item
      if (KIND == KIND_ANG) {
        if (s.p.angle < 0) build_projected_line(scratch, sm, s, s.p.is_ver ? sh.w : sh.h, s.p.is_ver ? sh.h : sh.w, gl, gsize);
      } else if (KIND == KIND_MIP) {
        if (!laneMip) build_mip_planes(scratch, scratch + mip_plane_offset(mg, sh), rom, sm, mg, sh, P.bd, s.mode, gl, gsize);
      } else {
        // DC value (CL/IntraPrediction.cpp:248-285), summed by the slot's lanes
        int part = 0;
        if (s.kind == 1) {
          const int16_t* top = sm.lines[s.set][0] + s.mrl + 1;
          const int16_t* left = sm.lines[s.set][1] + s.mrl + 1;
          if (sh.w >= sh.h) for (int i = gl; i < sh.w; i += gsize) part += top[i];
          if (sh.w <= sh.h) for (int i = gl; i < sh.h; i += gsize) part += left[i];
        }
        for (int o = gsize >> 1; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        const int denom = sh.w == sh.h ? 2 * sh.w : vmax(sh.w, sh.h);
        dc = (part + (denom >> 1)) >> vlog2(denom);
      }
      __syncwarp();

      int sad = 0, satd = 0;
      const bool transposed = KIND == KIND_ANG && !s.p.is_ver;
      MipSlot ms = {};
      int mipCarry[4] = {};
      if (laneMip) ms = make_mip_slot(sMip, mg, sm.mipIn, sm.mipAux, s.mode);
      if constexpr (S == 8) {
        // An 8x8 unit is processed as two 4x8 halves by the same loop body (kept rolled: the fully unrolled unit was
        // > 64 KB of code and instruction-fetch bound, profiles/r1m_summary.md history).  Rows and the first two column stages of the
        // Hadamard run inside a half; the column stage across the halves is folded into the absolute sum,
        // |a+b| + |a-b| = 2 max(|a|, |b|); for 16x8 / 8x16 tiles the stage across the two units of the tile is a real
        // butterfly with the partner lane.
        const int ux = u & (sh.unitsX - 1), uy = u >> sh.lgTilesX;
        const int x0 = ux * 8, y0 = uy * 8;
        const int partnerMask = TILE == 4 ? 1 : sh.unitsX;
        const bool owner = TILE == 4 ? (ux & 1) == 0 : (uy & 1) == 0;
        uint32_t c0[4][4];                     // |coefficients| of the first half, two per register
        int t = 0;
#pragma unroll 1
        for (int k = 0; k < 2; k++) {
          int q[4][8], d[4][8];
          const int hx = transposed ? x0 + 4 * k : x0, hy = transposed ? y0 : y0 + 4 * k;   // picture origin of the half
          if (KIND == KIND_ANG)      predict_angular<4, 8>(sm, scratch, s, sh, sFilt, P.bd, x0, y0, 4 * k, q);
          else if (KIND == KIND_MIP && laneMip) predict_mip_lane<TILE, 4, 8>(sm, ms, k, (1 << P.bd) - 1, mipCarry, q);
          else if (KIND == KIND_MIP) predict_mip<4, 8>(sm, scratch + mip_plane_offset(mg, sh), mg, sh, hx, hy, q);
          else pred_planar_dc_unit<4, 8>(sm.lines[s.set][0], sm.lines[s.set][1], s.kind, s.p.pdpc, dc, sh.lw, sh.lh, hx, hy, q);
          if (WITH_PRED && P.predOut && act) store_pred<4, 8>(P.predOut + (size_t)slot * sh.w * sh.h, sh.w, hx, hy, transposed, q);
          if (transposed) residual_unit<4, 8, true>(org + hy * P.stride + hx, P.stride, q, d, sad);
          else            residual_unit<4, 8, false>(org + hy * P.stride + hx, P.stride, q, d, sad);
          wht_rows_rc<4, 8>(d);
          wht_cols_rc<4, 8>(d);
          if (TILE != 3) {
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
        if (TILE == 3) satd = (2 * t + 2) >> 2;                                // CL/RdCost.cpp:2306
        else {
          t += __shfl_xor_sync(0xffffffffu, t, partnerMask);
          satd = owner ? satd_norm_rect(2 * t, true) : 0;                      // CL/RdCost.cpp:2452, :2589
        }
      } else {
        // 4xN / Nx4 shapes: a lane owns one SATD tile = one (4x4) or two (8x4, 4x8) 4x4 units
        const int tx = u & ((1 << sh.lgTilesX) - 1), ty = u >> sh.lgTilesX;
        uint32_t c0[4][2];                     // |coefficients| of the first 4x4 unit of the tile, two per register
        int t = 0;
#pragma unroll
        for (int k = 0; k < (TILE == 0 ? 1 : 2); k++) {
          const int x0 = tx * (TILE == 1 ? 8 : 4) + (TILE == 1 ? 4 * k : 0);
          const int y0 = ty * (TILE == 2 ? 8 : 4) + (TILE == 2 ? 4 * k : 0);
          int q[4][4], d[4][4];
          if (KIND == KIND_ANG)      predict_angular<4, 4>(sm, scratch, s, sh, sFilt, P.bd, x0, y0, 0, q);
          else if (KIND == KIND_MIP && laneMip) predict_mip_lane<TILE, 4, 4>(sm, ms, k, (1 << P.bd) - 1, mipCarry, q);
          else if (KIND == KIND_MIP) predict_mip<4, 4>(sm, scratch + mip_plane_offset(mg, sh), mg, sh, x0, y0, q);
          else pred_planar_dc_unit<4, 4>(sm.lines[s.set][0], sm.lines[s.set][1], s.kind, s.p.pdpc, dc, sh.lw, sh.lh, x0, y0, q);
          if (WITH_PRED && P.predOut && act) store_pred<4, 4>(P.predOut + (size_t)slot * sh.w * sh.h, sh.w, x0, y0, transposed, q);
          if (transposed) residual_unit<4, 4, true>(org + y0 * P.stride + x0, P.stride, q, d, sad);
          else            residual_unit<4, 4, false>(org + y0 * P.stride + x0, P.stride, q, d, sad);
          wht_rows<4>(d);
          if (TILE == 0) {
            satd = (wht_cols_abs_sum<4>(d) + 1) >> 1;                       // CL/RdCost.cpp:2209
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
        if (TILE != 0) satd = satd_norm_rect(2 * t, false);                 // CL/RdCost.cpp:2662, :2741
      }
      if (!act) { sad = 0; satd = 0; }

      if (lanes <= 32) {
        for (int o = gsize >> 1; o > 0; o >>= 1) {
          sad  += __shfl_xor_sync(0xffffffffu, sad, o);
          satd += __shfl_xor_sync(0xffffffffu, satd, o);
        }
        if (act && gl == 0) {
          const size_t at = scratch_at(slot, vIdx, P.nVisits);
          if (P.satdSM) { P.sadSM[at] = (uint32_t)sad; P.satdSM[at] = (uint32_t)satd; }
          else P.sadSM[at] = (uint32_t)vmin(2 * sad, satd);                                          // EL/IntraSearch.cpp:515
        }
      } else {
        // 64 lanes per slot: two consecutive warp iterations belong to the same slot
        accSad += sad; accSatd += satd;
        if (((base >> 5) & 1) == 1) {
          for (int o = 16; o > 0; o >>= 1) {
            accSad  += __shfl_xor_sync(0xffffffffu, accSad, o);
            accSatd += __shfl_xor_sync(0xffffffffu, accSatd, o);
          }
          if (lane == 0) {
            const size_t at = scratch_at(slot, vIdx, P.nVisits);
            if (P.satdSM) { P.sadSM[at] = (uint32_t)accSad; P.satdSM[at] = (uint32_t)accSatd; }
            else P.sadSM[at] = (uint32_t)vmin(2 * accSad, accSatd);
          }
          accSad = 0; accSatd = 0;
        }
      }
    }
  }
  }
}

template <int TILE, int KIND, int MODE>
__global__ void __launch_bounds__(EvalCfg<MODE == 1>::kThreads, EvalCfg<MODE == 1>::kMinCtas) rmd_eval_kernel(EvalParams P)
{
  __shared__ EvalShared<MODE == 1> shm;
  if constexpr (kLaneMip<TILE, KIND, MODE>) {
    alignas(16) __shared__ uint32_t sMip[kMipLaneWords];
    rmd_eval_body<TILE, KIND, MODE>(P, shm, sMip);
  } else rmd_eval_body<TILE, KIND, MODE>(P, shm, nullptr);
}

// One launch for every bucket a walk-sized batch occupies (vvcb_cu_eval: a few dozen visits of mixed shapes): the CTAs of the grid are dealt
// to the (tile class, kind) buckets by a small table and each runs that bucket's body.  A batch of 40 CUs spent more device time between its
// ~16 evaluation launches than inside them (profiles/r2_summary.md); the sweep keeps the per-bucket kernels (their own register allocation).
struct EvalAny {
  int n;                       // buckets in this launch
  int firstCta[19];            // CTAs [firstCta[k], firstCta[k + 1]) serve bucket[k]
  unsigned char bucket[20];    // tile class * kNumKinds + kind
};

template <int MODE>
__global__ void __launch_bounds__(EvalCfg<MODE == 1>::kThreads, EvalCfg<MODE == 1>::kMinCtas) rmd_eval_any_kernel(EvalParams P, EvalAny A)
{
  __shared__ EvalShared<MODE == 1> shm;
  alignas(16) __shared__ uint32_t sMip[MODE == 0 ? 1 : kMipLaneWords];
  int k = 0;
  while (k + 1 < A.n && (int)blockIdx.x >= A.firstCta[k + 1]) k++;
  switch (A.bucket[k]) {
    case 0:  rmd_eval_body<0, 0, MODE>(P, shm, sMip); break;  case 1:  rmd_eval_body<0, 1, MODE>(P, shm, sMip); break;  case 2:  rmd_eval_body<0, 2, MODE>(P, shm, sMip); break;
    case 3:  rmd_eval_body<1, 0, MODE>(P, shm, sMip); break;  case 4:  rmd_eval_body<1, 1, MODE>(P, shm, sMip); break;  case 5:  rmd_eval_body<1, 2, MODE>(P, shm, sMip); break;
    case 6:  rmd_eval_body<2, 0, MODE>(P, shm, sMip); break;  case 7:  rmd_eval_body<2, 1, MODE>(P, shm, sMip); break;  case 8:  rmd_eval_body<2, 2, MODE>(P, shm, sMip); break;
    case 9:  rmd_eval_body<3, 0, MODE>(P, shm, sMip); break;  case 10: rmd_eval_body<3, 1, MODE>(P, shm, sMip); break;  case 11: rmd_eval_body<3, 2, MODE>(P, shm, sMip); break;
    case 12: rmd_eval_body<4, 0, MODE>(P, shm, sMip); break;  case 13: rmd_eval_body<4, 1, MODE>(P, shm, sMip); break;  case 14: rmd_eval_body<4, 2, MODE>(P, shm, sMip); break;
    case 15: rmd_eval_body<5, 0, MODE>(P, shm, sMip); break;  case 16: rmd_eval_body<5, 1, MODE>(P, shm, sMip); break;  case 17: rmd_eval_body<5, 2, MODE>(P, shm, sMip); break;
  }
}

// =====================================================================================================
// prediction + residual of TU jobs (the first half of IntraSearch::xIntraCodingTUBlock, EL/IntraSearch.cpp:2820-2925):
// initIntraPatternChType, predIntraAng / predIntraMip, resi = org - pred.  One warp per job; the lanes share the
// visit's reference lines and take the units of the block in turn.  Low volume (a handful of surviving modes per CU
// against ~100 evaluated ones), so all prediction kinds live in this one kernel.
// =====================================================================================================
struct TuPredParams {
  const vvcb_rmd_visit* visits;
  const vvcb_tu_src*    src;       // per job: which visit, which evaluation slot
  const vvcb_tu_job*    jobs;
  int                   n;
  int16_t*              pred;      // dense w*h blocks at job.offset
  int16_t*              resi;
  const int16_t*        orig;
  const int16_t*        reco;
  int                   stride, bd, ctu;
  const Rom*            rom;
};

constexpr int kTuPredWarps = 4;

__global__ void __launch_bounds__(kTuPredWarps * 32) tu_pred_kernel(TuPredParams P)
{
  __shared__ WarpSmem smem[kTuPredWarps];
  __shared__ int16_t sScratch[kTuPredWarps][kSlotLineWords];
  __shared__ uint32_t sFilt[64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpSmem& sm = smem[warp];
  int16_t* const slotBuf = sScratch[warp];
  if (threadIdx.x < 64) sFilt[threadIdx.x] = (&P.rom->filt[0][0])[threadIdx.x];
  __syncthreads();
  const Rom& rom = *P.rom;
  for (int ji = blockIdx.x * kTuPredWarps + warp; ji < P.n; ji += gridDim.x * kTuPredWarps) {
    const vvcb_tu_src src = P.src[ji];
    const vvcb_rmd_visit v = P.visits[src.visit];
    const Shape sh = make_shape(v.log2w, v.log2h);
    const MipGeom mg = make_mip_geom(sh.w, sh.h);
    const int slot = src.slot;
    const SlotInfo s = make_slot_info(rom, v, sh, slot);
    const int16_t* org = P.orig + (size_t)v.y * P.stride + v.x;
    int16_t* predOut = P.pred + P.jobs[ji].offset;
    int16_t* resiOut = P.resi + P.jobs[ji].offset;
    __syncwarp();
    build_line_set(sm, 0, 0, v, sh, P.reco, P.stride, P.bd, lane);
    if (s.mrl) build_line_set(sm, s.set, s.mrl, v, sh, P.reco, P.stride, P.bd, lane);
    __syncwarp();
    if (s.kind != 3) build_filtered_set(sm, sh, lane);
    else             build_mip_inputs(sm, sh, mg, P.bd, lane);
    __syncwarp();
    int dc = 0;
    if (s.kind == 2) {
      if (s.p.angle < 0) build_projected_line(slotBuf, sm, s, s.p.is_ver ? sh.w : sh.h, s.p.is_ver ? sh.h : sh.w, lane, 32);
    } else if (s.kind == 3) {
      build_mip_planes(slotBuf, slotBuf + mip_plane_offset(mg, sh), rom, sm, mg, sh, P.bd, s.mode, lane, 32);
    } else if (s.kind == 1) {
      int part = 0;
      const int16_t* top = sm.lines[s.set][0] + s.mrl + 1;
      const int16_t* left = sm.lines[s.set][1] + s.mrl + 1;
      if (sh.w >= sh.h) for (int i = lane; i < sh.w; i += 32) part += top[i];
      if (sh.w <= sh.h) for (int i = lane; i < sh.h; i += 32) part += left[i];
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      const int denom = sh.w == sh.h ? 2 * sh.w : vmax(sh.w, sh.h);
      dc = (part + (denom >> 1)) >> vlog2(denom);
    }
    __syncwarp();
    const bool transposed = s.kind == 2 && !s.p.is_ver;
    // 4x4 pieces of the block in raster order, one per lane and round (the same piece functions as the evaluation kernels)
    const int piecesX = sh.w >> 2, pieces = (sh.w * sh.h) >> 4;
    for (int u = lane; u < pieces; u += 32) {
      const int x0 = (u % piecesX) * 4, y0 = (u / piecesX) * 4;
      int q[4][4];
      if (s.kind == 2)      predict_angular<4, 4>(sm, slotBuf, s, sh, sFilt, P.bd, x0, y0, 0, q);
      else if (s.kind == 3) predict_mip<4, 4>(sm, slotBuf + mip_plane_offset(mg, sh), mg, sh, x0, y0, q);
      else pred_planar_dc_unit<4, 4>(sm.lines[s.set][0], sm.lines[s.set][1], s.kind, s.p.pdpc, dc, sh.lw, sh.lh, x0, y0, q);
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int by = transposed ? y0 + j : y0 + i, bx = transposed ? x0 + i : x0 + j;
          predOut[by * sh.w + bx] = (int16_t)q[i][j];
          resiOut[by * sh.w + bx] = (int16_t)(org[by * P.stride + bx] - q[i][j]);
        }
    }
  }
}

// =====================================================================================================
// intra sub-partitions (vvcb_isp_eval): prediction of block k of every candidate, one warp per candidate
// =====================================================================================================
// A candidate is one ISP CU x split x luma mode x quantiser setting; its blocks (2 or 4, all of one size, at least 4x4) are coded in
// order and block k is predicted from the reconstruction of block k-1 (EL/IntraSearch.cpp:3171 xIntraCodingLumaISP).  The reference
// builds the lines of block k > 0 by shifting the side it holds and re-fetching the line block k-1 has just reconstructed
// (initIntraPatternChTypeISP, CL/IntraPrediction.cpp:1136-1203).  This kernel makes the equivalent fresh fetch: the same padding walk as
// make_line_geom, with the lengths m_topRefLength / m_leftRefLength of the block and availability derived from the CU's -- which agrees
// with the shift for all-or-nothing left and above neighbours only (vvcb_isp_eval refuses the rest).  Samples inside the CU come from the
// candidate's own reconstruction buffer, the others from the picture.
struct IspCand {                   // host-built (vvcb_api.cu), one per candidate
  int16_t x, y, cuW, cuH;          // CU in the picture
  int16_t bw, bh, topLen, leftLen; // block size, reference-line lengths of every block
  uint8_t hor, nParts, availAl, nAbove, nAboveRight, nLeft, nBelowLeft, mode;
  uint32_t offset;                 // first sample of the candidate's blocks (coding order, each dense bw*bh)
  ModeParam p;                     // make_mode_param_isp
};
struct IspState {                  // per candidate, carried from step to step
  vvcb_bin_model ctx[2];           // Ctx::QtCbf[luma] contexts 2, 3
  uint32_t cbfBits[4];
  uint8_t cbf[4], anyCbf, pad[3];
};
struct IspPredParams {
  const IspCand* cands;
  const int* list; int n;          // candidates with a block k, and (k > 0) those whose last block is k - 1
  int k;
  vvcb_tu_job* jobs;               // step k's TU jobs, index = candidate: cbf_delta_bits is written here
  const vvcb_tu_result* prev;      // step k - 1's results
  IspState* state;
  int16_t* pred; int16_t* resi;
  const int16_t* cuReco;           // candidates' reconstructions (coding order, like pred)
  const int16_t* orig; const int16_t* reco; int stride, bd;
  const Rom* rom;
  const uint32_t* frac;            // ProbModelTables::m_binFracBits
};

// price and adapt one context-coded bin (TBitEstimator::encodeBin; the same arithmetic as rate_bin, vvcb_rate.cuh)
__device__ __forceinline__ uint32_t isp_code_bin(vvcb_bin_model& m, const uint32_t* frac, unsigned bin)
{
  const unsigned rate0 = m.rate >> 4, rate1 = m.rate & 15, s0 = m.state[0], s1 = m.state[1];
  const uint32_t bits = frac[2 * ((s0 + s1) >> 8) + bin];
  unsigned n0 = s0 - ((s0 >> rate0) & 0x7fe0u), n1 = s1 - ((s1 >> rate1) & 0x7ffeu);
  if (bin) { n0 += (0x7fffu >> rate0) & 0x7fe0u; n1 += (0x7fffu >> rate1) & 0x7ffeu; }
  m.state[0] = (uint16_t)n0; m.state[1] = (uint16_t)n1;
  return bits;
}

// [lo, hi) clipped to [0, n); empty -> kNoInterval
__device__ __forceinline__ void isp_interval(int lo, int hi, int n, int& a, int& b)
{
  lo = vmax(lo, 0); hi = vmin(hi, n);
  if (lo < hi) { a = lo; b = hi; } else { a = kNoInterval; b = kNoInterval; }
}

constexpr int kIspPredWarps = 4;

__global__ void __launch_bounds__(kIspPredWarps * 32) isp_pred_kernel(IspPredParams P)
{
  __shared__ WarpSmem smem[kIspPredWarps];
  __shared__ int16_t sScratch[kIspPredWarps][kSlotLineWords];
  __shared__ uint32_t sFilt[64];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  WarpSmem& sm = smem[warp];
  int16_t* const slotBuf = sScratch[warp];
  if (threadIdx.x < 64) sFilt[threadIdx.x] = (&P.rom->filt[0][0])[threadIdx.x];
  __syncthreads();
  const int k = P.k;
  for (int q = blockIdx.x * kIspPredWarps + warp; q < P.n; q += gridDim.x * kIspPredWarps) {
    const int c = P.list[q];
    const IspCand cd = P.cands[c];
    // ---- cbf of block k - 1, then cbfDeltaBits of block k (RateEstimator::xSetLastCoeffOffset, CL/DepQuant.cpp:491-540, ISP branch):
    // block j's cbf is coded with context 2 + cbf of block j - 1, except the last block's when every earlier one is 0 (inferred 1)
    if (lane == 0) {
      IspState st = P.state[c];
      if (k > 0) {
        const int j = k - 1;
        const unsigned cbf = P.prev[c].abs_sum_level != 0;
        const bool inferred = j == cd.nParts - 1 && !st.anyCbf;
        st.cbfBits[j] = inferred ? 0u : isp_code_bin(st.ctx[j ? st.cbf[j - 1] : 0], P.frac, cbf);
        st.cbf[j] = (uint8_t)cbf;
        st.anyCbf |= (uint8_t)cbf;
      }
      if (k < cd.nParts) {
        const bool inferred = k == cd.nParts - 1 && !st.anyCbf;
        const vvcb_bin_model m = st.ctx[k ? st.cbf[k - 1] : 0];
        const int qs = ((int)m.state[0] + (int)m.state[1]) >> 8;
        P.jobs[c].cbf_delta_bits = inferred ? 0 : (int32_t)P.frac[2 * qs + 1] - (int32_t)P.frac[2 * qs];
      }
      P.state[c] = st;
    }
    if (k >= cd.nParts) continue;                                   // finishing pass of a candidate: its last cbf only
    const bool hor = cd.hor != 0;
    const int bx = hor ? 0 : k * cd.bw, by = hor ? k * cd.bh : 0, bs = cd.bw * cd.bh;
    const int T = cd.topLen, L = cd.leftLen;
    VVCB_EMUL_ASSERT(T + 2 < kLineMax && L + 2 < kLineMax);          // the lines and their two replicated samples fit the line arrays
    // ---- walk of block k: left[L] .. left[1], corner, top[1] .. top[T]; availability intervals in walk order
    LineGeom g;
    g.w = T; g.h = L; g.mrl = 0; g.n = L + 1 + T;
    int a, b;
    if (k == 0 || hor) {                                            // the CU's left column, shifted by the block's row
      isp_interval(cd.cuH - by, cd.cuH + 4 * cd.nBelowLeft - by, L, a, b); g.lo[0] = a == kNoInterval ? a : L - b; g.hi[0] = a == kNoInterval ? a : L - a;
      isp_interval(-by, 4 * cd.nLeft - by, L, a, b);                   g.lo[1] = a == kNoInterval ? a : L - b; g.hi[1] = a == kNoInterval ? a : L - a;
    } else {                                                        // vertical split: block k-1's last column, nothing below the CU
      g.lo[0] = g.hi[0] = kNoInterval;
      isp_interval(0, cd.cuH, L, a, b);                               g.lo[1] = L - b; g.hi[1] = L - a;
    }
    const bool corner = k == 0 ? cd.availAl != 0 : (hor ? by - 1 < 4 * cd.nLeft : bx - 1 < 4 * cd.nAbove);
    g.lo[2] = corner ? L : kNoInterval; g.hi[2] = corner ? L + 1 : kNoInterval;
    if (k == 0 || !hor) {                                           // the CU's above row, shifted by the block's column
      isp_interval(-bx, 4 * cd.nAbove - bx, T, a, b);                  g.lo[3] = a == kNoInterval ? a : L + 1 + a; g.hi[3] = a == kNoInterval ? a : L + 1 + b;
      isp_interval(cd.cuW - bx, cd.cuW + 4 * cd.nAboveRight - bx, T, a, b); g.lo[4] = a == kNoInterval ? a : L + 1 + a; g.hi[4] = a == kNoInterval ? a : L + 1 + b;
    } else {                                                        // horizontal split: block k-1's last row, nothing right of the CU
      isp_interval(0, cd.cuW, T, a, b);                               g.lo[3] = L + 1 + a; g.hi[3] = L + 1 + b;
      g.lo[4] = g.hi[4] = kNoInterval;
    }
    g.first = -1;
#pragma unroll
    for (int t = 4; t >= 0; t--) if (g.lo[t] != kNoInterval) g.first = g.lo[t];
    const int16_t* cuReco = P.cuReco + cd.offset;
    __syncwarp();
    // walk positions, then the two replicated samples past each line's end (CL/IntraPrediction.cpp:717-726, refLength = the ISP lengths)
    for (int i = lane; i < g.n + 4; i += 32) {
      const int pos = i < g.n ? i : (i < g.n + 2 ? g.n - 1 : 0);
      const int src = line_source(g, pos);
      int val = 1 << (P.bd - 1);
      if (src >= 0) {
        const int px = src < L ? bx - 1 : (src == L ? bx - 1 : bx + src - L - 1);   // CU frame
        const int py = src < L ? by + L - 1 - src : by - 1;
        if (px >= 0 && py >= 0) {                                    // inside the CU: an earlier block of this candidate
          const int j = hor ? py / cd.bh : px / cd.bw;
          val = cuReco[j * bs + (py - (hor ? j * cd.bh : 0)) * cd.bw + px - (hor ? 0 : j * cd.bw)];
        } else val = P.reco[(size_t)(cd.y + py) * P.stride + cd.x + px];
      }
      if (i < L) sm.lines[0][1][L - i] = (int16_t)val;
      else if (i == L) { sm.lines[0][0][0] = (int16_t)val; sm.lines[0][1][0] = (int16_t)val; }
      else if (i < g.n) sm.lines[0][0][i - L] = (int16_t)val;
      else if (i < g.n + 2) sm.lines[0][0][T + 1 + i - g.n] = (int16_t)val;
      else sm.lines[0][1][L + 1 + i - g.n - 2] = (int16_t)val;
    }
    __syncwarp();
    // ---- prediction of the block: the units of tu_pred_kernel, unfiltered lines, cubic interpolation (make_mode_param_isp)
    const Shape sh = make_shape(vlog2(cd.bw), vlog2(cd.bh));
    SlotInfo s;
    s.mode = cd.mode; s.mrl = 0; s.set = 0; s.p = cd.p;
    s.kind = s.mode == 0 ? 0 : (s.mode == 1 ? 1 : 2);
    int dc = 0;
    if (s.kind == 2) {
      if (s.p.angle < 0) build_projected_line(slotBuf, sm, s, s.p.is_ver ? sh.w : sh.h, s.p.is_ver ? sh.h : sh.w, lane, 32);
    } else if (s.kind == 1) {
      int part = 0;
      const int16_t* top = sm.lines[0][0] + 1;
      const int16_t* left = sm.lines[0][1] + 1;
      if (sh.w >= sh.h) for (int i = lane; i < sh.w; i += 32) part += top[i];
      if (sh.w <= sh.h) for (int i = lane; i < sh.h; i += 32) part += left[i];
      for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      const int denom = sh.w == sh.h ? 2 * sh.w : vmax(sh.w, sh.h);
      dc = (part + (denom >> 1)) >> vlog2(denom);
    }
    __syncwarp();
    const bool transposed = s.kind == 2 && !s.p.is_ver;
    const int16_t* org = P.orig + (size_t)(cd.y + by) * P.stride + cd.x + bx;
    int16_t* predOut = P.pred + cd.offset + k * bs;
    int16_t* resiOut = P.resi + cd.offset + k * bs;
    const int piecesX = sh.w >> 2, pieces = (sh.w * sh.h) >> 4;
    for (int u = lane; u < pieces; u += 32) {
      const int x0 = (u % piecesX) * 4, y0 = (u / piecesX) * 4;
      int qv[4][4];
      if (s.kind == 2) predict_angular<4, 4>(sm, slotBuf, s, sh, sFilt, P.bd, x0, y0, 0, qv);
      else pred_planar_dc_unit<4, 4>(sm.lines[0][0], sm.lines[0][1], s.kind, s.p.pdpc, dc, sh.lw, sh.lh, x0, y0, qv);
#pragma unroll
      for (int i = 0; i < 4; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          const int yy = transposed ? y0 + j : y0 + i, xx = transposed ? x0 + i : x0 + j;
          predOut[yy * sh.w + xx] = (int16_t)qv[i][j];
          resiOut[yy * sh.w + xx] = (int16_t)(org[yy * P.stride + xx] - qv[i][j]);
        }
    }
  }
}

// calls F<TILE, KIND, MODE>(args) for launch b = tile class * kNumKinds + kind
#define VVCB_FOR_BUCKET(b, PACK, F, ...)                                                                    \
  switch (b) {                                                                                               \
    case 0:  F<0, 0, PACK>(__VA_ARGS__); break;  case 1:  F<0, 1, PACK>(__VA_ARGS__); break;  case 2:  F<0, 2, PACK>(__VA_ARGS__); break; \
    case 3:  F<1, 0, PACK>(__VA_ARGS__); break;  case 4:  F<1, 1, PACK>(__VA_ARGS__); break;  case 5:  F<1, 2, PACK>(__VA_ARGS__); break; \
    case 6:  F<2, 0, PACK>(__VA_ARGS__); break;  case 7:  F<2, 1, PACK>(__VA_ARGS__); break;  case 8:  F<2, 2, PACK>(__VA_ARGS__); break; \
    case 9:  F<3, 0, PACK>(__VA_ARGS__); break;  case 10: F<3, 1, PACK>(__VA_ARGS__); break;  case 11: F<3, 2, PACK>(__VA_ARGS__); break; \
    case 12: F<4, 0, PACK>(__VA_ARGS__); break;  case 13: F<4, 1, PACK>(__VA_ARGS__); break;  case 14: F<4, 2, PACK>(__VA_ARGS__); break; \
    case 15: F<5, 0, PACK>(__VA_ARGS__); break;  case 16: F<5, 1, PACK>(__VA_ARGS__); break;  case 17: F<5, 2, PACK>(__VA_ARGS__); break; \
  }

// =====================================================================================================
// candidate lists
// =====================================================================================================
// g_aucIntraModeNumFast_UseMPM_2D, CL/Rom.cpp:536
__constant__ uint8_t cFastModes[6][6] = {
  { 3, 3, 3, 3, 2, 2 }, { 3, 3, 3, 3, 3, 2 }, { 3, 3, 3, 3, 3, 2 }, { 3, 3, 3, 3, 3, 2 }, { 2, 3, 3, 3, 3, 2 }, { 2, 2, 2, 2, 2, 3 } };

constexpr int kListThreads = 128;

// Scratch planes -> per-visit detail tables (only when the caller asked for details), through a shared-memory tile (written for the
// slot-major layout, where it was a transpose; with the visit-major planes it is a staged copy that fills the slots never evaluated).
__global__ void __launch_bounds__(256) rmd_detail_kernel(const vvcb_rmd_visit* visits, int n, int ctu, vvcb_rmd_detail* details,
                                                         const uint32_t* sadSM, const uint32_t* satdSM)
{
  __shared__ uint32_t tile[32][2 * VVCB_NUM_SLOTS + 1];
  const int first = blockIdx.x * 32;
  const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
  const int vi = first + lane;
  if (vi < n) {
    const vvcb_rmd_visit v = visits[vi];
    const bool mrlAllowed = visit_mrl_allowed(v, ctu);
    const int numMip = visit_num_mip(v);
    for (int s = wrp; s < VVCB_NUM_SLOTS; s += 8) {
      const bool evaluated = s < VVCB_SLOT_MRL1 || (s < VVCB_SLOT_MIP ? mrlAllowed : s - VVCB_SLOT_MIP < numMip);
      tile[lane][s] = evaluated ? sadSM[scratch_at(s, (unsigned)vi, n)] : VVCB_SAT_NONE;
      tile[lane][VVCB_NUM_SLOTS + s] = evaluated ? satdSM[scratch_at(s, (unsigned)vi, n)] : VVCB_SAT_NONE;
    }
  }
  __syncthreads();
  for (int r = wrp; r < 32 && first + r < n; r += 8) {
    uint32_t* dst = details[first + r].sad;          // sad[112] and satd[112] are contiguous
    for (int k = lane; k < 2 * VVCB_NUM_SLOTS; k += 32) dst[k] = tile[r][k];
  }
}

// ---- candidate lists in shared memory: entry i of thread t lives at [i * kListThreads + t] (conflict-free, and no
// per-thread local-memory arrays: an early profile (history in profiles/r1m_summary.md) showed the local-memory version waiting on the long scoreboard)
constexpr int kRdCap = VVCB_MAX_LIST + 2, kHadCap = VVCB_MAX_HAD_LIST;

struct SmList { uint32_t* m; double* c; int n; };

// vvcb_mode {mip, mrl, mode, pad} as one little-endian word
__device__ __forceinline__ uint32_t pack_mode(int mip, int mrl, int mode) { return (uint32_t)mip | ((uint32_t)mrl << 8) | ((uint32_t)mode << 16); }

// The same list in registers while the slots are being pushed (profiles/r1z_summary.md: the shared-memory insertion loops were 55 % of the
// kernel's instructions and its threads diverge on them).  Fixed capacity CAP, every step statically indexed.  A list of cap entries
// fills the last cap slots: the slots in front hold kPad, below any cost, and slots not filled yet hold +inf.  So the last kept cost is
// always c[CAP - 1] (the common case -- no better than anything kept -- is one comparison), an insertion is one compare and two
// selects per slot, and the cap grows by one with a static shift (reg_grow).
constexpr double kPad = -1.0;                     // costs are sums of non-negative terms
template <int CAP> struct RegList { uint32_t m[CAP]; double c[CAP]; };

template <int CAP> __device__ __forceinline__ void reg_init(RegList<CAP>& L, int cap)
{
#pragma unroll
  for (int i = 0; i < CAP; i++) { L.m[i] = 0u; L.c[i] = i < CAP - cap ? kPad : INFINITY; }
}

// updateCandList (CL/UnitTools.h:261-307): stable bounded insertion, strict '<'.  Slot i takes slot i - 1 when the cost goes in front
// of both, the cost when it goes in front of slot i only; ties keep the earlier entry, the last slot falls off.
template <int CAP> __device__ __forceinline__ void reg_push(RegList<CAP>& L, uint32_t m, double cost)
{
  if (!(cost < L.c[CAP - 1])) return;
  bool lt[CAP];
#pragma unroll
  for (int i = 0; i < CAP; i++) lt[i] = cost < L.c[i];
#pragma unroll
  for (int i = CAP - 1; i >= 1; i--) {
    L.m[i] = lt[i - 1] ? L.m[i - 1] : (lt[i] ? m : L.m[i]);
    L.c[i] = lt[i - 1] ? L.c[i - 1] : (lt[i] ? cost : L.c[i]);
  }
  if (lt[0]) { L.m[0] = m; L.c[0] = cost; }
}

// cap -> cap + 1 (needs cap < CAP): the list moves one slot to the front over a pad, the new last slot is empty.  Entries dropped
// under the smaller cap stay dropped.
template <int CAP> __device__ __forceinline__ void reg_grow(RegList<CAP>& L)
{
#pragma unroll
  for (int i = 0; i < CAP - 1; i++) { L.m[i] = L.m[i + 1]; L.c[i] = L.c[i + 1]; }
  L.m[CAP - 1] = 0u; L.c[CAP - 1] = INFINITY;
}

// the kept entries, from the front of the shared-memory list
template <int CAP> __device__ __forceinline__ void reg_to_sm(const RegList<CAP>& R, SmList& L)
{
  int n = 0;
#pragma unroll
  for (int i = 0; i < CAP; i++)
    if (R.c[i] != kPad && R.c[i] != INFINITY) { L.m[n * kListThreads] = R.m[i]; L.c[n * kListThreads] = R.c[i]; n++; }
  L.n = n;
}

__device__ void store_list_detail(const SmList& L, int32_t* n, vvcb_mode* m, double* c, int cap)
{
  *n = L.n;
  for (int i = 0; i < cap; i++) {
    reinterpret_cast<uint32_t*>(m)[i] = i < L.n ? L.m[i * kListThreads] : 0u;
    c[i] = i < L.n ? L.c[i * kListThreads] : 0.0;
  }
}

// One thread per visit: EL/IntraSearch.cpp:489-802 minus the predictions (already reduced to SAD/SATD, read from
// the visit's 448 contiguous bytes of the scratch plane, scratch_at: mostly L2 hits, the evaluation kernels have just written them).
// The result structs are written by the whole warp, one visit after the other, so that every store is a full line.
#ifndef VVCB_LIST_MIN_CTAS
#define VVCB_LIST_MIN_CTAS 4
#endif
__global__ void __launch_bounds__(kListThreads, VVCB_LIST_MIN_CTAS) rmd_lists_kernel(const vvcb_rmd_visit* visits, int n, int ctu, vvcb_rmd_result* results,
                                                                 vvcb_rmd_detail* details, const uint32_t* sadSM, const uint32_t* satdSM, vvcb_rmd_brief* brief)
{
  __shared__ double   sRdC[kRdCap * kListThreads], sHadC[kHadCap * kListThreads];
  __shared__ uint32_t sRdM[kRdCap * kListThreads], sHadM[kHadCap * kListThreads];
  __shared__ int      sCount[3 * kListThreads];              // n_rd, n_had, n_final per thread
  __shared__ uint8_t  sParent[8 * kListThreads];
  const int tid = threadIdx.x;
  const int vi = blockIdx.x * blockDim.x + tid;
  const bool live = vi < n;
  SmList rd, had;
  rd.m = sRdM + tid; rd.c = sRdC + tid; rd.n = 0;
  had.m = sHadM + tid; had.c = sHadC + tid; had.n = 0;
  constexpr int kRegRd = 9, kRegHad = 6;                     // K + 1 <= 9 (64x64 with MIP), numHad <= 6
  RegList<kRegRd> rrd; RegList<kRegHad> rhad;
  if (live) {
    const vvcb_rmd_visit v = visits[vi];
    const int w = 1 << v.log2w, h = 1 << v.log2h;
    const bool mipEnabled = !(v.flags & VVCB_VISIT_NO_MIP);
    const int numMip = visit_num_mip(v);
    const bool testMip = numMip > 0;
    const bool mrlAllowed = visit_mrl_allowed(v, ctu);
    const uint32_t* mySad = sadSM;
    const uint32_t* mySatd = satdSM;                                // nullptr: sadSM already holds min(2 * SAD, SATD)
    vvcb_rmd_detail* D = details ? details + vi : nullptr;

    auto dist_of = [&](int slot) -> double {
      const size_t at = scratch_at(slot, (unsigned)vi, n);
      if (!mySatd) return (double)mySad[at];
      const uint64_t sad = mySad[at], satd = mySatd[at];
      return (double)(sad * 2 < satd ? sad * 2 : satd);                        // :515
    };
    auto cost_of = [&](double dist, bool isMip, int mrl, int mode) -> double {
      const uint64_t bits = mode_bits(v.rates, v.mpm, w, h, mrlAllowed, mipEnabled, isMip, mrl, mode);
      return __dadd_rn(dist, __dmul_rn((double)bits, v.sqrt_lambda));          // :526, no FMA contraction
    };

    int K = cFastModes[v.log2w - 2][v.log2h - 2];
    if (testMip) K += vmax(K, vlog2(vmin(w, h)) - 1);                          // :472
    const int numHad = testMip ? 6 : 3;
    reg_init(rrd, K); reg_init(rhad, numHad);
    uint64_t checked0 = 0, checked1 = 0;                                       // bSatdChecked
    for (int m = 0; m < VVCB_NUM_LUMA_MODE; m++) {                             // :489-532
      if (m > 1 && (m & 1)) continue;
      if (m < 64) checked0 |= 1ull << m; else checked1 |= 1ull << (m - 64);
      const double dist = dist_of(m);
      reg_push(rrd, pack_mode(0, 0, m), cost_of(dist, false, 0, m));
      reg_push(rhad, pack_mode(0, 0, m), dist);
    }
#pragma unroll
    for (int i = kRegRd - 8; i < kRegRd; i++) if (i >= kRegRd - K) sParent[(i - (kRegRd - K)) * kListThreads + tid] = (uint8_t)(rrd.m[i] >> 16);
    for (int i = 0; i < K; i++) {                                              // :577-623
      const int pm = sParent[i * kListThreads + tid];
      if (pm > 2 && pm < 66)
        for (int dlt = -1; dlt <= 1; dlt += 2) {
          const int m = pm + dlt;
          const bool done = m < 64 ? (checked0 >> m) & 1 : (checked1 >> (m - 64)) & 1;
          if (done) continue;
          const double dist = dist_of(m);
          reg_push(rrd, pack_mode(0, 0, m), cost_of(dist, false, 0, m));
          reg_push(rhad, pack_mode(0, 0, m), dist);
          if (m < 64) checked0 |= 1ull << m; else checked1 |= 1ull << (m - 64);
        }
    }
    if (mrlAllowed)                                                            // :635-681
      for (int li = 0; li < 2; li++)
        for (int i = 1; i < 6; i++) {
          const int slot = (li ? VVCB_SLOT_MRL3 : VVCB_SLOT_MRL1) + i - 1;
          const int mrl = li ? 3 : 1;
          const double dist = dist_of(slot);
          reg_push(rrd, pack_mode(0, mrl, v.mpm[i]), cost_of(dist, false, mrl, v.mpm[i]));
          reg_push(rhad, pack_mode(0, mrl, v.mpm[i]), dist);
        }
    if (D) {
      reg_to_sm(rrd, rd); reg_to_sm(rhad, had);
      store_list_detail(rd, &D->n_reg, D->reg_mode, D->reg_cost, VVCB_MAX_LIST);
      store_list_detail(had, &D->n_reg_had, D->reg_had_mode, D->reg_had_cost, VVCB_MAX_HAD_LIST);
    }

    if (testMip) {                                                             // :704-751
      double c3[6];                                                            // costs of MIP modes 3,4,5 and their transposes
#pragma unroll
      for (int i = 0; i < 6; i++) c3[i] = 0.0;
      const int off = numMip / 2;
      reg_grow(rrd);                                                           // cap K + 1
      for (int m = 0; m < numMip; m++) {
        const int slot = VVCB_SLOT_MIP + m;
        const double dist = dist_of(slot);
        const double c = cost_of(dist, true, 0, m);
#pragma unroll
        for (int i = 0; i < 3; i++) { if (m == 3 + i) c3[i] = c; if (m == 3 + i + off) c3[3 + i] = c; }
        reg_push(rrd, pack_mode(1, 0, m), c);
        reg_push(rhad, pack_mode(1, 0, m), __dmul_rn(0.8, dist));
      }
      reg_to_sm(rrd, rd); reg_to_sm(rhad, had);           // the rest edits the lists in place (dynamic positions)
      // reduceHadCandList, :4333-4405 (compacted in place: the write index never passes the read index)
      const double thr = __dadd_rn(1.0, __ddiv_rn(1.4, __dsqrt_rn((double)(w * h))));
      const int maxPerType = K >> 1;
      const double minCost = rd.c[0];
      bool keepOne = rd.n > K;
      int numConv = 0, numMipKept = 0, wn = 0;
      for (int idx = 0; idx < rd.n - (keepOne ? 0 : 1); idx++) {      // the bound follows keepOne, as in the reference
        const uint32_t mm = rd.m[idx * kListThreads];
        const double cc = rd.c[idx * kListThreads];
        bool add;
        if (!(mm & 0xff)) { add = numConv < 3; numConv += add; }
        else {
          add = numMipKept < maxPerType || cc < __dmul_rn(thr, minCost) || keepOne;
          keepOne = false;
          numMipKept += add;
        }
        if (add) { rd.m[wn * kListThreads] = mm; rd.c[wn * kListThreads] = cc; wn++; }
      }
      rd.n = wn;
      if (w > 8 && h > 8) {
        // the three MIP modes 3..5 (or their transposes), cheapest first (stable), first one not yet in the list (FastMIP)
        double sc[3]; uint32_t smm[3];
#pragma unroll
        for (int i = 0; i < 3; i++) {
          const bool tr = c3[3 + i] < c3[i];
          sc[i] = tr ? c3[3 + i] : c3[i];
          smm[i] = pack_mode(1, 0, tr ? 3 + i + off : 3 + i);
        }
        unsigned picked = 0;
        const int baseN = rd.n;
        for (int r = 0; r < 3; r++) {
          int best = -1;
#pragma unroll
          for (int i = 0; i < 3; i++)
            if (!((picked >> i) & 1) && (best < 0 || sc[i] < (best == 0 ? sc[0] : best == 1 ? sc[1] : sc[2]))) best = i;
          picked |= 1u << best;
          const uint32_t cand = best == 0 ? smm[0] : best == 1 ? smm[1] : smm[2];
          bool inc = false;
          for (int i = 0; i < baseN; i++) inc = inc || rd.m[i * kListThreads] == cand;
          if (!inc) { rd.m[rd.n * kListThreads] = cand; rd.c[rd.n * kListThreads] = 0.0; rd.n++; break; }
        }
      }
      K = rd.n;
    } else {
      reg_to_sm(rrd, rd); reg_to_sm(rhad, had);
    }
    sCount[tid] = rd.n;
    sCount[kListThreads + tid] = had.n;
    for (int i = 0; i < v.num_mpm_cand; i++) {                                 // :777-802
      const uint32_t mp = pack_mode(0, 0, v.mpm[i]);
      bool inc = false;
      for (int j = 0; j < K; j++) inc = inc || mp == rd.m[j * kListThreads];
      if (!inc) { rd.m[rd.n * kListThreads] = mp; rd.c[rd.n * kListThreads] = 0.0; rd.n++; K++; }
    }
    sCount[2 * kListThreads + tid] = rd.n;
  }
  __syncwarp();
  // ---- cooperative, coalesced store of the warp's 32 result structs (92 words each)
  const int lane = tid & 31, wbase = tid & ~31;
  constexpr int kWords = (int)(sizeof(vvcb_rmd_result) / 4);
  static_assert(sizeof(vvcb_rmd_result) == 368, "result layout");
  if (brief) {
    // brief records: 16 words per visit, the warp's 32 records are 512 consecutive words
    static_assert(sizeof(vvcb_rmd_brief) == 64, "brief layout");
    const int vis0 = blockIdx.x * blockDim.x + wbase;
    uint32_t* dst = reinterpret_cast<uint32_t*>(brief + vis0);
    auto code = [](uint32_t m) -> uint32_t { return ((m >> 16) & 0xff) | (((m >> 8) & 0xff) << 8) | ((m & 1) << 15); };   // pack_mode -> modeId | mRefId << 8 | mipFlg << 15
    for (int k = lane; k < 32 * 16; k += 32) {
      const int r = k >> 4, wd = k & 15, t = wbase + r;
      if (vis0 + r >= n) break;
      const int nRd = sCount[t], nHad = sCount[kListThreads + t], nFinal = sCount[2 * kListThreads + t];
      uint32_t val = 0;
      if (wd == 0) val = (uint32_t)nRd | (uint32_t)nHad << 8 | (uint32_t)nFinal << 16;
      else if (wd < 9) { const int i = 2 * (wd - 1); if (i < nFinal) val = code(sRdM[i * kListThreads + t]); if (i + 1 < nFinal) val |= code(sRdM[(i + 1) * kListThreads + t]) << 16; }
      else if (wd < 13) { const int i = 2 * (wd - 9); if (i < nHad) val = code(sHadM[i * kListThreads + t]); if (i + 1 < nHad) val |= code(sHadM[(i + 1) * kListThreads + t]) << 16; }
      dst[k] = val;
    }
  }
  if (results)
  for (int r = 0; r < 32; r++) {
    const int t = wbase + r;
    const int vis = blockIdx.x * blockDim.x + t;
    if (vis >= n) break;
    const int nRd = sCount[t], nHad = sCount[kListThreads + t], nFinal = sCount[2 * kListThreads + t];
    uint32_t* dst = reinterpret_cast<uint32_t*>(results + vis);
    for (int k = lane; k < kWords; k += 32) {
      uint32_t val = 0;
      if (k < 4) val = k == 0 ? nRd : k == 1 ? nHad : k == 2 ? nFinal : 0;
      else if (k < 20) { const int i = k - 4; if (i < nRd) val = sRdM[i * kListThreads + t]; }
      else if (k < 52) {
        const int i = (k - 20) >> 1;
        if (i < nRd) { const unsigned long long b = (unsigned long long)__double_as_longlong(sRdC[i * kListThreads + t]); val = (k & 1) ? (uint32_t)(b >> 32) : (uint32_t)b; }
      }
      else if (k < 60) { const int i = k - 52; if (i < nHad) val = sHadM[i * kListThreads + t]; }
      else if (k < 76) {
        const int i = (k - 60) >> 1;
        if (i < nHad) { const unsigned long long b = (unsigned long long)__double_as_longlong(sHadC[i * kListThreads + t]); val = (k & 1) ? (uint32_t)(b >> 32) : (uint32_t)b; }
      }
      else { const int i = k - 76; if (i < nFinal) val = sRdM[i * kListThreads + t]; }
      dst[k] = val;
    }
  }
}

}  // namespace
