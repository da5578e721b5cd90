// vvc_intra_b200 -- the C ABI of include/vvc_intra_b200.h: context, plane management and kernel launches.
// The kernels live in vvcb_rmd.cuh.  There is no CPU fallback anywhere in this library.
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <math.h>
#include <new>
#include "vvcb_rmd.cuh"
#include "vvcb_tu.cuh"
#include "vvcb_feat.cuh"
#include "vvcb_dq.cuh"
#include "vvcb_rate.cuh"
#include <vector>
#include <algorithm>
#include <time.h>
#include <thread>
#include <atomic>
#include "vvcb_romfill.h"

// =====================================================================================================
// integer-issue microbenchmark (roofline denominator; not part of the encoder path)
// =====================================================================================================
template <int KIND>   // 0: IMAD only, 1: IADD3/LOP3 only, 2: 1:1 mix
__global__ void __launch_bounds__(256) int_peak_kernel(const int* in, int* out, int iters)
{
  int a[8], b[8];
  const int k0 = in[threadIdx.x & 31], k1 = in[32 + (threadIdx.x & 31)];
#pragma unroll
  for (int i = 0; i < 8; i++) { a[i] = k0 + i; b[i] = k1 - i; }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int r = 0; r < 4; r++) {
#pragma unroll
      for (int i = 0; i < 8; i++) {
        if (KIND == 0)      { a[i] = a[i] * k1 + k0; b[i] = b[i] * k0 + k1; }
        else if (KIND == 1) { a[i] = (a[i] + k1) ^ k0; b[i] = (b[i] ^ k1) + k0; }   // IADD3 + LOP3 pairs
        else                { a[i] = a[i] * k1 + k0; b[i] = (b[i] + k1) ^ k0; }
      }
    }
  }
  int s = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) s += a[i] ^ b[i];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

// =====================================================================================================
// C ABI
// =====================================================================================================
constexpr int kSideStreams = 7;
// Scratch slots of a context: device (vvcb_ctx::dTu, tu_buf) and page-locked (vvcb_ctx::hPin, pin_buf).  The stage-1 arenas of
// vvcb_cu_eval and the arenas of vvcb_isp_eval share kStageIn / kStageOut: a context serves one call at a time.
enum TuSlot {
  kTuIn, kTuOut,                 // tu_eval_impl / vvcb_residual_bits: inputs from the host, outputs (+ dequantised coefficients)
  kTuResi, kTuCoeff,             // residual, transform coefficients (vvcb_tu_eval's want_coeff)
  kDqCoeff, kDqTabs, kDqScratch, kDqLists,   // quantiser scratch (quant_scratch)
  kStageIn, kStageOut,
  kTuSlots
};
enum PinSlot { kPinTuIn, kPinTuOut, kPinStageIn, kPinStageOut, kPinSlots };
struct vvcb_ctx {
  int device, bd, ctu;
  cudaStream_t stream;
  cudaEvent_t ev0, ev1;
  Rom* dRom;
  TrRom* dTrRom;
  void* dTu[kTuSlots]; size_t capTu[kTuSlots];
  DqRom* dDqRom;
  RateRom* dRateRom;
  int depQuant;                     // slice->getDepQuantEnabledFlag() (vvcb_set_option), 1 = the shipped configuration
  float tuMs[4]; int tuTimed; cudaEvent_t tev[5];   // per-kernel timing of vvcb_tu_eval: transform pass, dependent quantisation, reconstruction pass
  void* dFeat[2]; size_t capFeat[2]; // feature scratch: jobs / per-CTU sums, results
  // copy/compute pipeline of vvcb_rmd_eval for large host batches
  cudaStream_t sIn, sOut; cudaEvent_t evIn[2], evComp[2], evOut[2];
  cudaStream_t sKind[kSideStreams]; cudaEvent_t evPlan, evKind[kSideStreams];   // evaluation launches are dealt over the main stream and these: the CTAs of the next kernels fill the tail of each one
  int evalStreams;                  // streams in use (1 + side streams), VVCB_EVAL_STREAMS for A/B runs
  vvcb_rmd_visit* dVisP[2]; vvcb_rmd_result* dResP[2]; bool pipeReady;
  vvcb_rmd_brief* dBrief; size_t capBrief;   // brief records of the un-pipelined path (the pipeline re-uses dResP)
  int trusted;                      // VVCB_OPT_TRUSTED_VISITS
  int16_t* dOrig; int16_t* dReco;
  const int16_t* bOrig; const int16_t* bReco;   // planes in use (own or bound)
  int width, height, stride;        // planes share one pitch (in samples)
  size_t planeSamples;
  // scratch for the host-pointer API
  vvcb_rmd_visit* dVisits; vvcb_rmd_result* dResults; size_t capVisits;
  vvcb_rmd_detail* dDetails; size_t capDetails;
  uint32_t* dScratch; size_t capScratch;   // SAD / SATD scratch: two planes of n * VVCB_NUM_SLOTS words, visit-major (scratch_at, vvcb_rmd.cuh)
  WorkItem* dItems; size_t capItems;
  PlanState* dPlan;
  int16_t* dPred; size_t capPred;
  int numSms;
  int16_t* wReco;                   // writable reconstruction plane: own (dReco) or another context's (vvcb_frame_share)
  int yieldSync; cudaEvent_t evYield;   // VVCB_OPT_YIELD_SYNC
  void* remote;                     // broker client proxy: VVCB_BROKER was set at vvcb_create (vvcb_broker.inc)
  void* hPin[kPinSlots]; size_t capPin[kPinSlots];
  void* dRect[2]; size_t capRect[2];
  uint64_t launches;
  uint64_t cuNs[8], cuCalls, tuWaitFrom;    // vvcb_cu_eval_phases
  cudaEvent_t cev[4]; bool cuSpan;          // device spans of the two stages of vvcb_cu_eval
  int timing; int timedLaunches; float kms[3]; cudaEvent_t kev[4];
  char err[512];
};

static char g_createErr[512] = "";

#define CK(call)                                                                                          \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) {                                                                              \
      snprintf(ctx->err, sizeof(ctx->err), "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return VVCB_ERR_CUDA;                                                                               \
    }                                                                                                     \
  } while (0)

// wait for the context's stream: polling (default) or, with VVCB_OPT_YIELD_SYNC, sleeping on a blocking event
static inline uint64_t host_ns() { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec; }

static cudaError_t ctx_sync(vvcb_ctx* ctx)
{
  if (!ctx->yieldSync) return cudaStreamSynchronize(ctx->stream);
  cudaError_t e = cudaEventRecord(ctx->evYield, ctx->stream);
  if (e != cudaSuccess) return e;
  if (ctx->yieldSync == 1) return cudaEventSynchronize(ctx->evYield);
  // value N >= 2: look every N microseconds and sleep in between (the blocking event's wake-up costs several hundred microseconds on some
  // hosts, tools/sync_latency.cu; a timed sleep of a real-time thread does not)
  timespec nap = { 0, (long)ctx->yieldSync * 1000 };
  while ((e = cudaEventQuery(ctx->evYield)) == cudaErrorNotReady) nanosleep(&nap, nullptr);
  return e;
}

#include "vvcb_broker.inc"

extern "C" int vvcb_device_count(void)
{
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

extern "C" const char* vvcb_last_error(const vvcb_ctx* ctx) { return ctx ? ctx->err : g_createErr; }

extern "C" void vvcb_destroy(vvcb_ctx* ctx);

extern "C" int vvcb_create(vvcb_ctx** out, int device, int bit_depth, int ctu_size)
{
  // bit depths above 10 would need the negative transform-skip shift branch of TrQuant::xTransformSkip (CL/TrQuant.cpp:1394) and have no
  // golden coverage: refused rather than computed differently.  H.266 caps CtbSizeY at 128 (sps_log2_ctu_size_minus5 <= 2).
  if (!out || bit_depth < 8 || bit_depth > 10 || ctu_size < 32 || ctu_size > 128 || (ctu_size & (ctu_size - 1))) {
    snprintf(g_createErr, sizeof(g_createErr), "vvcb_create: bad argument (bit depth 8..10, CTU size 32, 64 or 128)");
    return VVCB_ERR_ARG;
  }
  *out = nullptr;
  if (const char* path = getenv("VVCB_BROKER")) {         // this process is a walker: the engine lives in the broker's server process
    vvcb_ctx* ctx = new (std::nothrow) vvcb_ctx();
    if (!ctx) return VVCB_ERR_ARG;
    memset(ctx, 0, sizeof(*ctx));
    ctx->device = -1; ctx->bd = bit_depth; ctx->ctu = ctu_size; ctx->depQuant = 1;
    ctx->remote = vvcbc_connect(path, bit_depth, ctu_size, g_createErr, sizeof(g_createErr));
    if (!ctx->remote) { delete ctx; return VVCB_ERR_STATE; }
    *out = ctx;
    return VVCB_OK;
  }
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || device < 0 || device >= n) {
    snprintf(g_createErr, sizeof(g_createErr), "vvcb_create: no usable CUDA device %d (%s); this library has no CPU path",
             device, e != cudaSuccess ? cudaGetErrorString(e) : "index out of range");
    return VVCB_ERR_CUDA;
  }
  vvcb_ctx* ctx = new (std::nothrow) vvcb_ctx();
  if (!ctx) return VVCB_ERR_ARG;
  memset(ctx, 0, sizeof(*ctx));
  ctx->device = device; ctx->bd = bit_depth; ctx->ctu = ctu_size; ctx->depQuant = 1;
  auto fail = [&](const char* what, cudaError_t err) {
    snprintf(g_createErr, sizeof(g_createErr), "vvcb_create: %s: %s", what, cudaGetErrorString(err));
    vvcb_destroy(ctx);                       // releases whatever was created so far (the context is zero-initialised)
    return VVCB_ERR_CUDA;
  };
  if ((e = cudaSetDevice(device)) != cudaSuccess) return fail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return fail("cudaGetDeviceProperties", e);
  ctx->numSms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
  {
    const char* env = getenv("VVCB_EVAL_STREAMS");
    const int v = env ? atoi(env) : 0;
    ctx->evalStreams = v >= 1 && v <= kSideStreams + 1 ? v : kSideStreams + 1;
  }
  for (int i = 0; i < kSideStreams; i++) {
    if ((e = cudaStreamCreateWithFlags(&ctx->sKind[i], cudaStreamNonBlocking)) != cudaSuccess) return fail("cudaStreamCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->evKind[i], cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  }
  if ((e = cudaEventCreateWithFlags(&ctx->evPlan, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&ctx->evYield, cudaEventBlockingSync | cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
  if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return fail("cudaEventCreate", e);
  for (int i = 0; i < 4; i++) if ((e = cudaEventCreate(&ctx->kev[i])) != cudaSuccess) return fail("cudaEventCreate", e);
  for (int i = 0; i < 4; i++) if ((e = cudaEventCreate(&ctx->cev[i])) != cudaSuccess) return fail("cudaEventCreate", e);
  for (int i = 0; i < 5; i++) if ((e = cudaEventCreate(&ctx->tev[i])) != cudaSuccess) return fail("cudaEventCreate", e);
  Rom* h = new Rom();
  fill_rom(*h);
  if ((e = cudaMalloc(&ctx->dRom, sizeof(Rom))) != cudaSuccess) { delete h; return fail("cudaMalloc(rom)", e); }
  e = cudaMemcpy(ctx->dRom, h, sizeof(Rom), cudaMemcpyHostToDevice);
  delete h;
  if (e != cudaSuccess) return fail("cudaMemcpy(rom)", e);
  if ((e = cudaMalloc(&ctx->dPlan, sizeof(PlanState))) != cudaSuccess) return fail("cudaMalloc(plan)", e);
  {
    TrRom* t = new TrRom();
    fill_tr_rom(*t);
    if ((e = cudaMalloc(&ctx->dTrRom, sizeof(TrRom))) != cudaSuccess) { delete t; return fail("cudaMalloc(trrom)", e); }
    e = cudaMemcpy(ctx->dTrRom, t, sizeof(TrRom), cudaMemcpyHostToDevice);
    delete t;
    if (e != cudaSuccess) return fail("cudaMemcpy(trrom)", e);
  }
  {
    DqRom* t = new DqRom();
    fill_dq_rom(*t);
    if ((e = cudaMalloc(&ctx->dDqRom, sizeof(DqRom))) != cudaSuccess) { delete t; return fail("cudaMalloc(dqrom)", e); }
    e = cudaMemcpy(ctx->dDqRom, t, sizeof(DqRom), cudaMemcpyHostToDevice);
    delete t;
    if (e != cudaSuccess) return fail("cudaMemcpy(dqrom)", e);
  }
  {
    RateRom t;
    for (int i = 0; i < 512; i++) t.binFracBits[i] = kBinFracBits[i];
    if ((e = cudaMalloc(&ctx->dRateRom, sizeof(RateRom))) != cudaSuccess) return fail("cudaMalloc(raterom)", e);
    if ((e = cudaMemcpy(ctx->dRateRom, &t, sizeof(RateRom), cudaMemcpyHostToDevice)) != cudaSuccess) return fail("cudaMemcpy(raterom)", e);
  }
  *out = ctx;
  return VVCB_OK;
}

extern "C" void vvcb_destroy(vvcb_ctx* ctx)
{
  if (!ctx) return;
  if (ctx->remote) { vvcbc_disconnect(ctx->remote); delete ctx; return; }
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < kPinSlots; i++) if (ctx->hPin[i]) cudaFreeHost(ctx->hPin[i]);
  cudaFree(ctx->dRect[0]); cudaFree(ctx->dRect[1]); cudaFree(ctx->dBrief);
  cudaFree(ctx->dRom); cudaFree(ctx->dOrig); cudaFree(ctx->dReco); cudaFree(ctx->dVisits); cudaFree(ctx->dResults); cudaFree(ctx->dDetails); cudaFree(ctx->dScratch);
  cudaFree(ctx->dItems); cudaFree(ctx->dPlan); cudaFree(ctx->dPred); cudaFree(ctx->dTrRom);
  for (int i = 0; i < kTuSlots; i++) cudaFree(ctx->dTu[i]);
  cudaFree(ctx->dRateRom);
  cudaFree(ctx->dDqRom);
  for (int i = 0; i < 2; i++) cudaFree(ctx->dFeat[i]);
  if (ctx->pipeReady) {
    cudaStreamSynchronize(ctx->sIn); cudaStreamSynchronize(ctx->sOut);
    for (int i = 0; i < 2; i++) { cudaFree(ctx->dVisP[i]); cudaFree(ctx->dResP[i]); cudaEventDestroy(ctx->evIn[i]); cudaEventDestroy(ctx->evComp[i]); cudaEventDestroy(ctx->evOut[i]); }
    cudaStreamDestroy(ctx->sIn); cudaStreamDestroy(ctx->sOut);
  }
  cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1); cudaEventDestroy(ctx->evYield);
  for (int i = 0; i < 4; i++) cudaEventDestroy(ctx->kev[i]);
  for (int i = 0; i < 4; i++) cudaEventDestroy(ctx->cev[i]);
  for (int i = 0; i < 5; i++) cudaEventDestroy(ctx->tev[i]);
  for (int i = 0; i < kSideStreams; i++) { cudaStreamSynchronize(ctx->sKind[i]); cudaStreamDestroy(ctx->sKind[i]); cudaEventDestroy(ctx->evKind[i]); }
  cudaEventDestroy(ctx->evPlan);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

extern "C" int vvcb_set_option(vvcb_ctx* ctx, int option, int value)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (option == VVCB_OPT_DEP_QUANT && (value == 0 || value == 1)) {
    ctx->depQuant = value;
    return ctx->remote ? vvcbc_set_option(ctx->remote, option, value, ctx->err, sizeof(ctx->err)) : VVCB_OK;
  }
  if (option == VVCB_OPT_YIELD_SYNC && value >= 0 && value <= 1000) { ctx->yieldSync = value; return VVCB_OK; }
  if (option == VVCB_OPT_TRUSTED_VISITS && (value == 0 || value == 1)) { ctx->trusted = value; return VVCB_OK; }
  snprintf(ctx->err, sizeof(ctx->err), "vvcb_set_option: unknown option %d or bad value %d", option, value);
  return VVCB_ERR_ARG;
}

extern "C" int vvcb_frame_begin(vvcb_ctx* ctx, const int16_t* orig, int stride, int width, int height)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (!orig || width <= 0 || height <= 0 || stride < width || (width & 3) || (height & 3)) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_frame_begin: bad argument (width/height must be positive multiples of 4)");
    return VVCB_ERR_ARG;
  }
  if (ctx->remote) return vvcbc_frame_begin(ctx->remote, orig, stride, width, height, ctx->err, sizeof(ctx->err));
  CK(cudaSetDevice(ctx->device));
  const int pitch = (width + 63) & ~63;
  const size_t samples = (size_t)pitch * height;
  if (samples > ctx->planeSamples) {
    cudaFree(ctx->dOrig); cudaFree(ctx->dReco);
    ctx->dOrig = ctx->dReco = nullptr; ctx->planeSamples = 0;
    CK(cudaMalloc(&ctx->dOrig, samples * sizeof(int16_t)));
    CK(cudaMalloc(&ctx->dReco, samples * sizeof(int16_t)));
    ctx->planeSamples = samples;
  }
  ctx->width = width; ctx->height = height; ctx->stride = pitch;
  ctx->bOrig = ctx->dOrig; ctx->bReco = ctx->dReco; ctx->wReco = ctx->dReco;
  CK(cudaMemcpy2DAsync(ctx->dOrig, pitch * sizeof(int16_t), orig, stride * sizeof(int16_t), width * sizeof(int16_t), height,
                       cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(ctx->dReco, 0, samples * sizeof(int16_t), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

#define REMOTE_UNAVAILABLE(name)                                                                                      \
  if (ctx->remote) { snprintf(ctx->err, sizeof(ctx->err), name ": not available through the broker"); return VVCB_ERR_STATE; }

extern "C" int vvcb_frame_alloc(vvcb_ctx* ctx, int width, int height)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_frame_alloc");
  if (width <= 0 || height <= 0 || (width & 3) || (height & 3)) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_frame_alloc: bad argument"); return VVCB_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  const int pitch = (width + 63) & ~63;
  const size_t samples = (size_t)pitch * height;
  if (samples > ctx->planeSamples) {
    cudaFree(ctx->dOrig); cudaFree(ctx->dReco);
    ctx->dOrig = ctx->dReco = nullptr; ctx->planeSamples = 0;
    CK(cudaMalloc(&ctx->dOrig, samples * sizeof(int16_t)));
    CK(cudaMalloc(&ctx->dReco, samples * sizeof(int16_t)));
    ctx->planeSamples = samples;
  }
  ctx->width = width; ctx->height = height; ctx->stride = pitch;
  ctx->bOrig = ctx->dOrig; ctx->bReco = ctx->dReco; ctx->wReco = ctx->dReco;
  CK(cudaMemsetAsync(ctx->dOrig, 0, samples * sizeof(int16_t), ctx->stream));
  CK(cudaMemsetAsync(ctx->dReco, 0, samples * sizeof(int16_t), ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_reco_from_orig(vvcb_ctx* ctx)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_reco_from_orig");
  if (!ctx->dReco || ctx->bReco != ctx->dReco || ctx->bOrig != ctx->dOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_from_orig: no frame owned by the context"); return VVCB_ERR_STATE; }
  CK(cudaSetDevice(ctx->device));
  // stream ordered: every later launch of this context (the pipelined path's kernels included) runs behind it
  CK(cudaMemcpyAsync(ctx->dReco, ctx->dOrig, (size_t)ctx->stride * ctx->height * sizeof(int16_t), cudaMemcpyDeviceToDevice, ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_frame_share(vvcb_ctx* dst, vvcb_ctx* src)
{
  if (!dst) return VVCB_ERR_ARG;
  vvcb_ctx* ctx = dst;
  REMOTE_UNAVAILABLE("vvcb_frame_share");
  if (!src || src->remote || !src->dOrig || src->bOrig != src->dOrig || src->device != dst->device) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_frame_share: the source context owns no frame on this device");
    return VVCB_ERR_STATE;
  }
  dst->bOrig = src->dOrig; dst->bReco = src->dReco; dst->wReco = src->dReco;
  dst->width = src->width; dst->height = src->height; dst->stride = src->stride;
  return VVCB_OK;
}

extern "C" int vvcb_orig_update(vvcb_ctx* ctx, const int16_t* orig, int stride, int x, int y, int w, int h)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_orig_update");
  if (!ctx->dOrig || ctx->bOrig != ctx->dOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_orig_update: no frame owned by the context"); return VVCB_ERR_STATE; }
  if (!orig || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > ctx->width || y + h > ctx->height || stride < w) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_orig_update: rectangle outside the picture");
    return VVCB_ERR_ARG;
  }
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy2DAsync(ctx->dOrig + (size_t)y * ctx->stride + x, ctx->stride * sizeof(int16_t), orig, stride * sizeof(int16_t),
                       w * sizeof(int16_t), h, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

// page-locked staging buffer i of at least `bytes`
static int pin_buf(vvcb_ctx* ctx, PinSlot i, size_t bytes)
{
  if (bytes > ctx->capPin[i]) {
    if (ctx->hPin[i]) cudaFreeHost(ctx->hPin[i]);
    ctx->hPin[i] = nullptr; ctx->capPin[i] = 0;
    const size_t cap = bytes + bytes / 2 + 4096;
    CK(cudaHostAlloc(&ctx->hPin[i], cap, cudaHostAllocDefault));
    ctx->capPin[i] = cap;
  }
  return VVCB_OK;
}

// Layout of one arena of several arrays: take() returns the next array's offset, 16-byte aligned (the kernels' widest access, uint4).
struct Arena {
  size_t size = 0;
  size_t take(size_t bytes) { const size_t at = size; size += (bytes + 15) & ~(size_t)15; return at; }
};
template <class T> static T* at(void* base, size_t offset) { return reinterpret_cast<T*>(static_cast<uint8_t*>(base) + offset); }

// one CTA per rectangle: dense w*h block -> the reconstruction plane
__global__ void __launch_bounds__(128) reco_scatter_kernel(const vvcb_rect* __restrict__ rects, int n, const int16_t* __restrict__ samples, int16_t* __restrict__ plane, int stride)
{
  for (int r = blockIdx.x; r < n; r += gridDim.x) {
    const vvcb_rect q = rects[r];
    const int16_t* src = samples + q.offset;
    int16_t* dst = plane + (size_t)q.y * stride + q.x;
    const int cnt = q.w * q.h;
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) { const int yy = i / q.w; dst[(size_t)yy * stride + (i - yy * q.w)] = src[i]; }
  }
}

// rectangles + samples are already validated and sit in host memory the copies may read asynchronously until the next sync
static int launch_reco_rects(vvcb_ctx* ctx, const vvcb_rect* rects, int n, const int16_t* samples, size_t n_samples)
{
  if (n == 0) return VVCB_OK;
  for (int i = 0; i < 2; i++) {
    const size_t need = i == 0 ? (size_t)n * sizeof(vvcb_rect) : n_samples * sizeof(int16_t);
    if (need > ctx->capRect[i]) {
      cudaFree(ctx->dRect[i]); ctx->dRect[i] = nullptr; ctx->capRect[i] = 0;
      CK(cudaMalloc(&ctx->dRect[i], need * 2));
      ctx->capRect[i] = need * 2;
    }
  }
  CK(cudaMemcpyAsync(ctx->dRect[0], rects, (size_t)n * sizeof(vvcb_rect), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(ctx->dRect[1], samples, n_samples * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
  reco_scatter_kernel<<<n < ctx->numSms * 8 ? n : ctx->numSms * 8, 128, 0, ctx->stream>>>(static_cast<const vvcb_rect*>(ctx->dRect[0]), n, static_cast<const int16_t*>(ctx->dRect[1]), ctx->wReco, ctx->stride);
  ctx->launches++;
  CK(cudaGetLastError());
  return VVCB_OK;
}

static bool rect_ok(const vvcb_ctx* ctx, const vvcb_rect& r, size_t n_samples)
{
  return r.x >= 0 && r.y >= 0 && r.w > 0 && r.h > 0 && r.x + r.w <= ctx->width && r.y + r.h <= ctx->height && (size_t)r.offset + (size_t)r.w * r.h <= n_samples;
}

extern "C" int vvcb_reco_update_rects(vvcb_ctx* ctx, const vvcb_rect* rects, int n, const int16_t* samples, size_t n_samples)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && (!rects || !samples))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update_rects: bad argument"); return VVCB_ERR_ARG; }
  if (ctx->remote) {
    vvcb_cu_request rq;
    memset(&rq, 0, sizeof(rq));
    rq.rects = rects; rq.n_rects = n; rq.rect_samples = samples; rq.n_rect_samples = n_samples;
    return vvcbc_cu_eval(ctx->remote, &rq, 1, ctx->err, sizeof(ctx->err));
  }
  if (!ctx->wReco || ctx->bReco != ctx->wReco) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update_rects: no writable frame (vvcb_frame_begin / vvcb_frame_alloc / vvcb_frame_share)"); return VVCB_ERR_STATE; }
  for (int i = 0; i < n; i++)
    if (!rect_ok(ctx, rects[i], n_samples)) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update_rects: rectangle %d is malformed or outside the picture", i); return VVCB_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  const int rc = launch_reco_rects(ctx, rects, n, samples, n_samples);
  if (rc) return rc;
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_reco_update(vvcb_ctx* ctx, const int16_t* reco, int stride, int x, int y, int w, int h)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) {
    if (!reco || w <= 0 || h <= 0 || stride < w) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update: bad argument"); return VVCB_ERR_ARG; }
    std::vector<int16_t> dense((size_t)w * h);
    for (int r = 0; r < h; r++) memcpy(&dense[(size_t)r * w], reco + (size_t)r * stride, (size_t)w * sizeof(int16_t));
    const vvcb_rect rc = { (int16_t)x, (int16_t)y, (int16_t)w, (int16_t)h, 0 };
    return vvcb_reco_update_rects(ctx, &rc, 1, dense.data(), dense.size());
  }
  if (!ctx->dReco || ctx->bReco != ctx->dReco) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update: no frame owned by the context"); return VVCB_ERR_STATE; }
  if (!reco || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > ctx->width || y + h > ctx->height || stride < w) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_reco_update: rectangle outside the picture");
    return VVCB_ERR_ARG;
  }
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpy2DAsync(ctx->dReco + (size_t)y * ctx->stride + x, ctx->stride * sizeof(int16_t), reco, stride * sizeof(int16_t),
                       w * sizeof(int16_t), h, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_frame_bind_device(vvcb_ctx* ctx, const void* d_orig, const void* d_reco, int stride, int width, int height)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_frame_bind_device");
  // the texture kernels read 8-sample rows as one 16-byte word: pitch a multiple of 8 samples, planes 16-byte aligned
  if (!d_orig || !d_reco || width <= 0 || height <= 0 || stride < width || (width & 3) || (height & 3) || (stride & 7) ||
      (reinterpret_cast<uintptr_t>(d_orig) & 15) || (reinterpret_cast<uintptr_t>(d_reco) & 15)) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_frame_bind_device: bad argument (stride must be a multiple of 8 samples, planes 16-byte aligned)");
    return VVCB_ERR_ARG;
  }
  ctx->bOrig = static_cast<const int16_t*>(d_orig); ctx->bReco = static_cast<const int16_t*>(d_reco); ctx->wReco = nullptr;
  ctx->width = width; ctx->height = height; ctx->stride = stride;
  return VVCB_OK;
}

extern "C" int vvcb_kernel_timing(vvcb_ctx* ctx, int on)
{
  if (!ctx) return VVCB_ERR_ARG;
  ctx->timing = on; ctx->timedLaunches = 0; ctx->kms[0] = ctx->kms[1] = ctx->kms[2] = 0.f;
  ctx->tuTimed = 0; ctx->tuMs[0] = ctx->tuMs[1] = ctx->tuMs[2] = ctx->tuMs[3] = 0.f;
  return VVCB_OK;
}

extern "C" int vvcb_kernel_times(vvcb_ctx* ctx, float ms[3], int* launches)
{
  if (!ctx || !ms) return VVCB_ERR_ARG;
  for (int i = 0; i < 3; i++) ms[i] = ctx->kms[i];
  if (launches) *launches = ctx->timedLaunches;
  ctx->timedLaunches = 0; ctx->kms[0] = ctx->kms[1] = ctx->kms[2] = 0.f;
  return VVCB_OK;
}

static int ensure_items(vvcb_ctx* ctx, int n)
{
  static_assert(kItemTasks >= 128, "the item bound below assumes at least 128 lane-tasks per plain work item");
  const size_t need = (size_t)n * 60 + 8; // worst case 64x64: three kinds, ceil(slots * 64 lanes / kItemTasks) items each
  if (need > ctx->capItems) {
    cudaFree(ctx->dItems); ctx->dItems = nullptr; ctx->capItems = 0;
    CK(cudaMalloc(&ctx->dItems, need * sizeof(WorkItem)));
    ctx->capItems = need;
  }
  return VVCB_OK;
}

static int ensure_details(vvcb_ctx* ctx, int n)
{
  if ((size_t)n > ctx->capDetails) {
    cudaFree(ctx->dDetails); ctx->dDetails = nullptr; ctx->capDetails = 0;
    CK(cudaMalloc(&ctx->dDetails, (size_t)n * sizeof(vvcb_rmd_detail)));
    ctx->capDetails = (size_t)n;
  }
  return VVCB_OK;
}

template <int TILE, int KIND, int MODE> static void launch_eval_bucket(const EvalParams& P, int numSms, long long maxWarps, cudaStream_t stream)
{
  using Cfg = EvalCfg<MODE == 1>;
  long long grid = (long long)numSms * Cfg::kMinCtas;
  const long long maxCtas = (maxWarps + Cfg::kWarps - 1) / Cfg::kWarps;
  if (grid > maxCtas) grid = maxCtas;
  if (grid < 1) grid = 1;
  rmd_eval_kernel<TILE, KIND, MODE><<<(int)grid, Cfg::kThreads, 0, stream>>>(P);
}

// hostVisits (optional): the same visits in host memory.  Small batches (the broker's: a handful of CUs per call) touch few of the 33
// (tile class, prediction kind, packed / plain) kernels; with the visits at hand the empty ones are not launched at all.
static int launch_rmd(vvcb_ctx* ctx, const vvcb_rmd_visit* dVisits, int n, vvcb_rmd_result* dResults, vvcb_rmd_detail* dDetails,
                      int16_t* dPred, const vvcb_rmd_visit* hostVisits = nullptr, vvcb_rmd_brief* dBrief = nullptr)
{
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  if (n == 0) return VVCB_OK;
  int rc = ensure_items(ctx, n);
  if (rc) return rc;
  if ((size_t)n > ctx->capScratch) {
    cudaFree(ctx->dScratch); ctx->dScratch = nullptr; ctx->capScratch = 0;
    CK(cudaMalloc(&ctx->dScratch, (size_t)n * 2 * VVCB_NUM_SLOTS * sizeof(uint32_t)));
    ctx->capScratch = (size_t)n;
  }
  const bool smallPlan = hostVisits && n <= 4096;         // walk-sized batch: one planning launch (rmd_plan_small), the plan state is written whole
  if (!smallPlan) CK(cudaMemsetAsync(ctx->dPlan, 0, sizeof(PlanState), ctx->stream));
  const bool tm = ctx->timing != 0;
  if (tm) CK(cudaEventRecord(ctx->kev[0], ctx->stream));
  const int pack = dPred ? 0 : 1;     // the prediction-output kernels (parity / integration entry points) take plain items only
  bool needAll = !hostVisits || n > 4096, need[2][kNumBuckets] = {};
  int inBucket[2][kNumBuckets] = {};                  // visits per (packed / plain, bucket)
  if (!needAll)
    for (int i = 0; i < n; i++) {
      const vvcb_rmd_visit& v = hostVisits[i];
      const Shape sh = make_shape(v.log2w, v.log2h);
      const int packed = pack && small_shape_index(sh.lw, sh.lh) >= 0 ? 1 : 0;
      const bool mip = !(v.flags & VVCB_VISIT_NO_MIP) && mip_num_modes(sh.w, sh.h) > 0;
      need[packed][sh.tile * kNumKinds + KIND_ANG] = need[packed][sh.tile * kNumKinds + KIND_PDC] = true;
      inBucket[packed][sh.tile * kNumKinds + KIND_ANG]++; inBucket[packed][sh.tile * kNumKinds + KIND_PDC]++;
      if (mip) { need[packed][sh.tile * kNumKinds + KIND_MIP] = true; inBucket[packed][sh.tile * kNumKinds + KIND_MIP]++; }
    }
  int evalLaunches = 0;
  if (smallPlan) rmd_plan_small<<<1, 256, 0, ctx->stream>>>(dVisits, n, ctx->ctu, ctx->dPlan, ctx->dItems, pack);
  else {
    rmd_plan_count<<<(n + 255) / 256, 256, 0, ctx->stream>>>(dVisits, n, ctx->ctu, ctx->dPlan, pack);
    rmd_plan_scan<<<1, 32, 0, ctx->stream>>>(ctx->dPlan);
    rmd_plan_fill<<<(n + 255) / 256, 256, 0, ctx->stream>>>(dVisits, n, ctx->ctu, ctx->dPlan, ctx->dItems, pack);
  }
  if (tm) CK(cudaEventRecord(ctx->kev[1], ctx->stream));
  EvalParams P;
  P.visits = dVisits; P.items = ctx->dItems; P.plan = ctx->dPlan;
  // without detail tables the lists only need min(2 * SAD, SATD): one scratch plane instead of two
  P.sadSM = ctx->dScratch; P.satdSM = (dDetails || dPred) ? ctx->dScratch + (size_t)VVCB_NUM_SLOTS * n : nullptr; P.nVisits = n;
  P.orig = ctx->bOrig; P.reco = ctx->bReco; P.stride = ctx->stride; P.bd = ctx->bd; P.ctu = ctx->ctu; P.rom = ctx->dRom;
  P.predOut = dPred;
  const long long maxWarps = (long long)n * 8;          // no point in more warps than work items
  // The launches are independent of each other (disjoint work items, disjoint scratch entries) and every grid fills the GPU.  Dealt over
  // several streams, longest first, the CTAs of the following kernels move in as soon as SM slots free up.  Measured (profiles/r1z_summary.md):
  // no effect on a whole resident sweep (persistent warps drain within one item of each other), 20.3 -> 17.7 ms for the chunked host-buffer
  // path, where every chunk pays the hand-over between its 33 launches.
  static const int kindOrder[kNumKinds] = { KIND_ANG, KIND_MIP, KIND_PDC };
  static const int tileOrder[kNumClasses] = { 3, 4, 5, 1, 2, 0 };
  if (!needAll && !dPred) {
    // walk-sized batch: ONE launch for the packed items and one for the plain ones, the CTAs dealt to the occupied buckets (rmd_eval_any_kernel)
    for (int mode = 1; mode >= 0; mode--) {
      EvalAny A;
      A.n = 0;
      int cta = 0;
      const int warpsPerCta = mode ? EvalCfg<true>::kWarps : EvalCfg<false>::kWarps, minCtas = mode ? EvalCfg<true>::kMinCtas : EvalCfg<false>::kMinCtas;
      for (int ki = 0; ki < kNumKinds; ki++)
        for (int ti = 0; ti < kNumClasses; ti++) {
          const int b = tileOrder[ti] * kNumKinds + kindOrder[ki];
          if (!need[mode][b] || (mode == 0 && b < kNumKinds)) continue;            // (the 4x4 class has no plain shapes)
          int ctas = (inBucket[mode][b] * 8 + warpsPerCta - 1) / warpsPerCta;     // no point in more warps than work items
          if (ctas > ctx->numSms * minCtas) ctas = ctx->numSms * minCtas;
          A.bucket[A.n] = (unsigned char)b; A.firstCta[A.n] = cta; cta += ctas; A.n++;
        }
      A.firstCta[A.n] = cta;
      if (!A.n) continue;
      if (mode) rmd_eval_any_kernel<1><<<cta, EvalCfg<true>::kThreads, 0, ctx->stream>>>(P, A);
      else      rmd_eval_any_kernel<0><<<cta, EvalCfg<false>::kThreads, 0, ctx->stream>>>(P, A);
      evalLaunches++;
    }
  } else {
  const int useStreams = needAll ? ctx->evalStreams : (ctx->evalStreams < 3 ? ctx->evalStreams : 3);   // a handful of launches: fewer hand-overs
  const int nSide = useStreams - 1;
  CK(cudaEventRecord(ctx->evPlan, ctx->stream));
  for (int i = 0; i < nSide; i++) CK(cudaStreamWaitEvent(ctx->sKind[i], ctx->evPlan, 0));
  int dealt = 0;
  auto next_stream = [&]() { const int k = dealt++ % useStreams; return k == 0 ? ctx->stream : ctx->sKind[k - 1]; };
  for (int ki = 0; ki < kNumKinds; ki++)
    for (int ti = 0; ti < kNumClasses; ti++) {
      const int b = tileOrder[ti] * kNumKinds + kindOrder[ki];
      if (dPred) { if (needAll || need[0][b]) { VVCB_FOR_BUCKET(b, 2, launch_eval_bucket, P, ctx->numSms, maxWarps, next_stream()); evalLaunches++; } continue; }
      // the packed small shapes of the tile class, and its larger shapes (the 4x4 class has none)
      if (needAll || need[1][b]) { VVCB_FOR_BUCKET(b, 1, launch_eval_bucket, P, ctx->numSms, maxWarps, next_stream()); evalLaunches++; }
      if (b >= kNumKinds && (needAll || need[0][b])) { VVCB_FOR_BUCKET(b, 0, launch_eval_bucket, P, ctx->numSms, maxWarps, next_stream()); evalLaunches++; }
    }
  for (int i = 0; i < nSide; i++) { CK(cudaEventRecord(ctx->evKind[i], ctx->sKind[i])); CK(cudaStreamWaitEvent(ctx->stream, ctx->evKind[i], 0)); }
  }
  if (tm) CK(cudaEventRecord(ctx->kev[2], ctx->stream));
  if (dDetails) { rmd_detail_kernel<<<(n + 31) / 32, 256, 0, ctx->stream>>>(dVisits, n, ctx->ctu, dDetails, P.sadSM, P.satdSM); ctx->launches++; }
  rmd_lists_kernel<<<(n + kListThreads - 1) / kListThreads, kListThreads, 0, ctx->stream>>>(dVisits, n, ctx->ctu, dResults, dDetails, P.sadSM, P.satdSM, dBrief);
  ctx->launches += (smallPlan ? 1 : 3) + evalLaunches + 1;
  CK(cudaGetLastError());
  if (tm) {
    CK(cudaEventRecord(ctx->kev[3], ctx->stream));
    CK(cudaEventSynchronize(ctx->kev[3]));
    for (int i = 0; i < 3; i++) { float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->kev[i], ctx->kev[i + 1])); ctx->kms[i] += ms; }
    ctx->timedLaunches++;
  }
  return VVCB_OK;
}

// The largest internal QP (6 * qp_per + qp_rem) of a luma block: 63 + QpBdOffset, QpBdOffset = 6 * (bitDepth - 8).
static int max_qp(int bd) { return 63 + 6 * (bd - 8); }
// lambda of the RD quantisers: the dependent quantiser derives shift counts from it (vvcb_dq.cuh, dq_init_quant), so +inf is refused too.
static bool lambda_ok(double l) { return l > 0.0 && isfinite(l); }

// Host-side validation of large batches runs on a few threads: returns the smallest index for which ok(i) is false, or -1.
template <class F> static int first_bad_index(int n, F ok)
{
  const int kMinPerThread = 32768;
  // a share of the host's cores: one process per GPU is the deployment (torchrun exports LOCAL_WORLD_SIZE), VVCB_HOST_THREADS overrides
  static int maxThreads = 0;
  if (!maxThreads) {
    int hc = (int)std::thread::hardware_concurrency();
    const char* e = getenv("VVCB_HOST_THREADS");
    const char* lw = getenv("LOCAL_WORLD_SIZE");
    int t = e ? atoi(e) : (lw && atoi(lw) > 1 ? hc / atoi(lw) : hc);
    maxThreads = t < 1 ? 1 : (t > 8 ? 8 : t);
  }
  int threads = maxThreads;
  if (threads < 1 || n < 2 * kMinPerThread) threads = 1;
  if (threads > n / kMinPerThread) threads = n / kMinPerThread > 0 ? n / kMinPerThread : 1;
  std::atomic<int> bad(n);
  auto work = [&](int lo, int hi) {
    for (int i = lo; i < hi && i < bad.load(std::memory_order_relaxed); i++)
      if (!ok(i)) { int cur = bad.load(); while (i < cur && !bad.compare_exchange_weak(cur, i)) {} break; }
  };
  if (threads == 1) work(0, n);
  else {
    std::vector<std::thread> pool;
    const int per = (n + threads - 1) / threads;
    for (int t = 0; t < threads; t++) pool.emplace_back(work, t * per, (t + 1) * per < n ? (t + 1) * per : n);
    for (auto& th : pool) th.join();
  }
  const int b = bad.load();
  return b < n ? b : -1;
}

static int check_visits(vvcb_ctx* ctx, const vvcb_rmd_visit* v, int n, int first = 0)
{
  if (ctx->trusted) return VVCB_OK;
  const int badIdx = first_bad_index(n, [&](int i) {
    const int w = 1 << v[i].log2w, h = 1 << v[i].log2h;
    const bool ok = v[i].log2w >= 2 && v[i].log2w <= 6 && v[i].log2h >= 2 && v[i].log2h <= 6 && v[i].x >= 0 && v[i].y >= 0 &&
                    (v[i].x & 3) == 0 && (v[i].y & 3) == 0 && v[i].x + w <= ctx->width && v[i].y + h <= ctx->height &&
                    v[i].n_above <= w / 4 && v[i].n_above_right <= w / 4 && v[i].n_left <= h / 4 && v[i].n_below_left <= h / 4 &&
                    v[i].avail_al <= 1 && v[i].num_mpm_cand <= 6 &&
                    // available samples must lie inside the picture
                    (!(v[i].avail_al || v[i].n_above || v[i].n_above_right) || v[i].y >= 4) &&
                    (!(v[i].avail_al || v[i].n_left || v[i].n_below_left) || v[i].x >= 4) &&
                    v[i].x + w + 4 * v[i].n_above_right <= ctx->width && v[i].y + h + 4 * v[i].n_below_left <= ctx->height;
    bool mpmOk = true;
    for (int k = 0; k < 6; k++) mpmOk = mpmOk && v[i].mpm[k] < VVCB_NUM_LUMA_MODE;
    return ok && mpmOk;
  });
  if (badIdx >= 0) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: visit %d is malformed (position/size/availability outside the picture)", first + badIdx);
    return VVCB_ERR_ARG;
  }
  return VVCB_OK;
}

static int ensure_visit_buffers(vvcb_ctx* ctx, int n)
{
  if ((size_t)n > ctx->capVisits) {
    cudaFree(ctx->dVisits); cudaFree(ctx->dResults);
    ctx->dVisits = nullptr; ctx->dResults = nullptr; ctx->capVisits = 0;
    CK(cudaMalloc(&ctx->dVisits, (size_t)n * sizeof(vvcb_rmd_visit)));
    CK(cudaMalloc(&ctx->dResults, (size_t)n * sizeof(vvcb_rmd_result)));
    ctx->capVisits = (size_t)n;
  }
  return VVCB_OK;
}

// Large host batches: the batch is cut into chunks and the three stages -- visits host->device, the kernels, result lists
// device->host -- run on three streams with double-buffered chunk storage, so that the PCIe copies and the host-side
// validation of the next chunk hide behind the kernels of the current one.
constexpr int kPipeChunkDefault = 172032;
// VVCB_PIPE_CHUNK (visits per chunk) is a tuning aid for the A/B runs in profiles/; read once
static int pipe_chunk()
{
  static int chunk = 0;
  if (!chunk) {
    const char* e = getenv("VVCB_PIPE_CHUNK");
    const long v = e ? atol(e) : 0;
    chunk = v >= 4096 && v <= (1 << 22) ? (int)v : kPipeChunkDefault;
  }
  return chunk;
}

static int ensure_pipeline(vvcb_ctx* ctx)
{
  if (ctx->pipeReady) return VVCB_OK;
  CK(cudaStreamCreateWithFlags(&ctx->sIn, cudaStreamNonBlocking));
  CK(cudaStreamCreateWithFlags(&ctx->sOut, cudaStreamNonBlocking));
  for (int i = 0; i < 2; i++) {
    CK(cudaEventCreateWithFlags(&ctx->evIn[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->evComp[i], cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&ctx->evOut[i], cudaEventDisableTiming));
    CK(cudaMalloc(&ctx->dVisP[i], (size_t)pipe_chunk() * sizeof(vvcb_rmd_visit)));
    CK(cudaMalloc(&ctx->dResP[i], (size_t)pipe_chunk() * sizeof(vvcb_rmd_result)));
  }
  ctx->pipeReady = true;
  return VVCB_OK;
}

// results or brief (exactly one): the record the chunks copy back
// dResident (optional): the visits already live on the device (a static plan such as the exhaustive sweep's): nothing is uploaded or validated
static int rmd_eval_pipelined(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_result* results, vvcb_rmd_brief* brief = nullptr,
                              const vvcb_rmd_visit* dResident = nullptr)
{
  int rc = ensure_pipeline(ctx);
  if (rc) return rc;
  const int savedTiming = ctx->timing;
  ctx->timing = 0;                                   // per-kernel timing would serialise the pipeline
  int status = VVCB_OK;
  // Chunk schedule: a short first chunk (the kernels start after a fraction of a millisecond of copying) and a short last one (the
  // copy of its results is all that is left when the kernels end); VVCB_PIPE_EDGE for A/B runs.
  const int chunk = pipe_chunk();
  static int edge = -1;
  if (edge < 0) { const char* e = getenv("VVCB_PIPE_EDGE"); const long v = e ? atol(e) : 0; edge = e && v >= 0 && v <= chunk ? (int)v : chunk / 4; }
  for (int c = 0, off = 0, m = 0; off < n && status == VVCB_OK; c++, off += m) {
    const int rest = n - off, b = c & 1;
    m = rest < chunk ? rest : chunk;
    if (edge > 0) {
      if (c == 0 && rest > edge) m = edge;
      else if (rest > edge && rest - m < edge) m = rest - edge;      // leave exactly one short chunk for the end
    }
    if (!dResident && (status = check_visits(ctx, visits + off, m, off))) break;
    cudaError_t e = cudaSuccess;
    const vvcb_rmd_visit* dIn = dResident ? dResident + off : ctx->dVisP[b];
    if (!dResident) {
      if (c >= 2) e = cudaStreamWaitEvent(ctx->sIn, ctx->evComp[b], 0);              // chunk c-2 no longer reads this buffer
      if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->dVisP[b], visits + off, (size_t)m * sizeof(vvcb_rmd_visit), cudaMemcpyHostToDevice, ctx->sIn);
      if (e == cudaSuccess) e = cudaEventRecord(ctx->evIn[b], ctx->sIn);
      if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->stream, ctx->evIn[b], 0);
    }
    if (e == cudaSuccess && c >= 2) e = cudaStreamWaitEvent(ctx->stream, ctx->evOut[b], 0);   // its results have left the device
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: pipeline stage failed: %s", cudaGetErrorString(e)); status = VVCB_ERR_CUDA; break; }
    // brief records are written into the chunk's result buffer (a fifth of its size)
    if ((status = brief ? launch_rmd(ctx, dIn, m, nullptr, nullptr, nullptr, nullptr, reinterpret_cast<vvcb_rmd_brief*>(ctx->dResP[b]))
                        : launch_rmd(ctx, dIn, m, ctx->dResP[b], nullptr, nullptr))) break;
    e = cudaEventRecord(ctx->evComp[b], ctx->stream);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(ctx->sOut, ctx->evComp[b], 0);
    if (e == cudaSuccess) e = brief ? cudaMemcpyAsync(brief + off, ctx->dResP[b], (size_t)m * sizeof(vvcb_rmd_brief), cudaMemcpyDeviceToHost, ctx->sOut)
                                    : cudaMemcpyAsync(results + off, ctx->dResP[b], (size_t)m * sizeof(vvcb_rmd_result), cudaMemcpyDeviceToHost, ctx->sOut);
    if (e == cudaSuccess) e = cudaEventRecord(ctx->evOut[b], ctx->sOut);
    if (e != cudaSuccess) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: pipeline stage failed: %s", cudaGetErrorString(e)); status = VVCB_ERR_CUDA; }
  }
  ctx->timing = savedTiming;
  // drain in every case: the caller owns the host buffers again when this returns
  cudaError_t e1 = cudaStreamSynchronize(ctx->sIn), e2 = cudaStreamSynchronize(ctx->stream), e3 = cudaStreamSynchronize(ctx->sOut);
  if (status == VVCB_OK && (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess)) {
    const cudaError_t e = e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3);
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: %s", cudaGetErrorString(e));
    status = VVCB_ERR_CUDA;
  }
  return status;
}

extern "C" int vvcb_rmd_eval(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_result* results, vvcb_rmd_detail* details)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && (!visits || !results))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  if (ctx->remote) {
    std::vector<vvcb_cu_request> rq(n);
    memset(rq.data(), 0, (size_t)n * sizeof(vvcb_cu_request));
    for (int i = 0; i < n; i++) { rq[i].visit = &visits[i]; rq[i].want_rmd = 1; rq[i].result = &results[i]; rq[i].detail = details ? &details[i] : nullptr; }
    return vvcbc_cu_eval(ctx->remote, rq.data(), n, ctx->err, sizeof(ctx->err));
  }
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  CK(cudaSetDevice(ctx->device));
  if (n > pipe_chunk() && !details) return rmd_eval_pipelined(ctx, visits, n, results);
  int rc = check_visits(ctx, visits, n);
  if (rc) return rc;
  rc = ensure_visit_buffers(ctx, n);
  if (rc) return rc;
  CK(cudaMemcpyAsync(ctx->dVisits, visits, (size_t)n * sizeof(vvcb_rmd_visit), cudaMemcpyHostToDevice, ctx->stream));
  if (details) {
    rc = ensure_details(ctx, n);
    if (rc) return rc;
  }
  rc = launch_rmd(ctx, ctx->dVisits, n, ctx->dResults, details ? ctx->dDetails : nullptr, nullptr);
  if (rc) return rc;
  CK(cudaMemcpyAsync(results, ctx->dResults, (size_t)n * sizeof(vvcb_rmd_result), cudaMemcpyDeviceToHost, ctx->stream));
  if (details) CK(cudaMemcpyAsync(details, ctx->dDetails, (size_t)n * sizeof(vvcb_rmd_detail), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_rmd_eval_brief(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_brief* out)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_rmd_eval_brief");
  if (n < 0 || (n > 0 && (!visits || !out))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval_brief: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval_brief: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  CK(cudaSetDevice(ctx->device));
  if (n > pipe_chunk()) return rmd_eval_pipelined(ctx, visits, n, nullptr, out);
  int rc = check_visits(ctx, visits, n);
  if (rc) return rc;
  if ((rc = ensure_visit_buffers(ctx, n))) return rc;
  if ((size_t)n > ctx->capBrief) {
    cudaFree(ctx->dBrief); ctx->dBrief = nullptr; ctx->capBrief = 0;
    CK(cudaMalloc(&ctx->dBrief, (size_t)n * sizeof(vvcb_rmd_brief)));
    ctx->capBrief = (size_t)n;
  }
  CK(cudaMemcpyAsync(ctx->dVisits, visits, (size_t)n * sizeof(vvcb_rmd_visit), cudaMemcpyHostToDevice, ctx->stream));
  if ((rc = launch_rmd(ctx, ctx->dVisits, n, nullptr, nullptr, nullptr, nullptr, ctx->dBrief))) return rc;
  CK(cudaMemcpyAsync(out, ctx->dBrief, (size_t)n * sizeof(vvcb_rmd_brief), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_rmd_eval_brief_resident(vvcb_ctx* ctx, const void* d_visits, int n, vvcb_rmd_brief* out)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_rmd_eval_brief_resident");
  if (n < 0 || (n > 0 && (!d_visits || !out))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval_brief_resident: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval_brief_resident: no frame"); return VVCB_ERR_STATE; }
  CK(cudaSetDevice(ctx->device));
  return rmd_eval_pipelined(ctx, nullptr, n, nullptr, out, static_cast<const vvcb_rmd_visit*>(d_visits));
}

extern "C" int vvcb_rmd_eval_device(vvcb_ctx* ctx, const void* d_visits, int n, void* d_results, void* d_details)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_rmd_eval_device");
  if (n < 0 || (n > 0 && (!d_visits || !d_results))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_eval_device: bad argument"); return VVCB_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  return launch_rmd(ctx, static_cast<const vvcb_rmd_visit*>(d_visits), n, static_cast<vvcb_rmd_result*>(d_results),
                    static_cast<vvcb_rmd_detail*>(d_details), nullptr);
}

// slot >= 0: the prediction of that slot (w*h samples); slot < 0: all VVCB_NUM_SLOTS predictions back to back (slots the visit does
// not evaluate are left untouched)
static int rmd_pred_impl(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int slot, int16_t* pred)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_rmd_pred");
  if (!visit || !pred || slot >= VVCB_NUM_SLOTS) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_pred: bad argument"); return VVCB_ERR_ARG; }
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_pred: no frame"); return VVCB_ERR_STATE; }
  int rc = check_visits(ctx, visit, 1);
  if (rc) return rc;
  const int w = 1 << visit->log2w, h = 1 << visit->log2h;
  const bool mrlAllowed = !(visit->flags & VVCB_VISIT_NO_MRL) && (visit->y & (ctx->ctu - 1)) != 0;
  const int numMip = (visit->flags & VVCB_VISIT_NO_MIP) ? 0 : mip_num_modes(w, h);
  if (slot >= 0) {
    const bool evaluated = slot < VVCB_SLOT_MRL1 || (slot < VVCB_SLOT_MIP ? mrlAllowed : slot - VVCB_SLOT_MIP < numMip);
    if (!evaluated) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_pred: slot %d is not evaluated for this visit", slot); return VVCB_ERR_ARG; }
  }
  CK(cudaSetDevice(ctx->device));
  rc = ensure_visit_buffers(ctx, 1);
  if (rc) return rc;
  const size_t need = (size_t)VVCB_NUM_SLOTS * w * h;
  if (need > ctx->capPred) {
    cudaFree(ctx->dPred); ctx->dPred = nullptr; ctx->capPred = 0;
    CK(cudaMalloc(&ctx->dPred, need * sizeof(int16_t)));
    ctx->capPred = need;
  }
  CK(cudaMemcpyAsync(ctx->dVisits, visit, sizeof(vvcb_rmd_visit), cudaMemcpyHostToDevice, ctx->stream));
  rc = launch_rmd(ctx, ctx->dVisits, 1, ctx->dResults, nullptr, ctx->dPred);
  if (rc) return rc;
  if (slot >= 0) CK(cudaMemcpyAsync(pred, ctx->dPred + (size_t)slot * w * h, (size_t)w * h * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
  else {
    // only the slots the visit evaluates: the device buffer holds an earlier visit's samples in the others, and the caller's copy of
    // those is left untouched (vvc_intra_b200.h)
    const int spans[3][2] = { { 0, VVCB_SLOT_MRL1 }, { VVCB_SLOT_MRL1, mrlAllowed ? VVCB_SLOT_MIP : VVCB_SLOT_MRL1 }, { VVCB_SLOT_MIP, VVCB_SLOT_MIP + numMip } };
    for (const auto& s : spans)
      if (s[1] > s[0])
        CK(cudaMemcpyAsync(pred + (size_t)s[0] * w * h, ctx->dPred + (size_t)s[0] * w * h, (size_t)(s[1] - s[0]) * w * h * sizeof(int16_t),
                           cudaMemcpyDeviceToHost, ctx->stream));
  }
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_rmd_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int slot, int16_t* pred)
{
  if (ctx && slot < 0) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_rmd_pred: bad argument"); return VVCB_ERR_ARG; }
  return rmd_pred_impl(ctx, visit, slot, pred);
}

extern "C" int vvcb_rmd_pred_all(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int16_t* pred) { return rmd_pred_impl(ctx, visit, -1, pred); }

// Walk mode of the TU stage (vvcb_cu_eval): every host input travels in ONE page-locked arena and every output comes back in one, both moved
// by a copy KERNEL over the mapped host memory instead of by the copy engines.  The engines' queues are shared by all streams of the
// process in issue order: the small copies of one broker worker waited there behind another worker's copy whose kernels were still
// running (0.6-0.7 ms per wait, profiles/r2_summary.md).  A kernel launch is ordered by its own stream only.
struct TuWalk {
  bool wantLevel, wantReco, wantPred;
  vvcb_tu_result* results; int32_t* level; int16_t* reco; int16_t* pred;      // out: where the results lie in the page-locked arena (valid until the next call)
};

__global__ void arena_copy_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, size_t n16)
{
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

static cudaError_t arena_copy(vvcb_ctx* ctx, const void* src, void* dst, size_t bytes)
{
  const size_t n16 = (bytes + 15) / 16;
  if (!n16) return cudaSuccess;
  const int grid = (int)std::min<size_t>((n16 + 255) / 256, (size_t)ctx->numSms * 4);
  arena_copy_kernel<<<grid, 256, 0, ctx->stream>>>(static_cast<const uint4*>(src), static_cast<uint4*>(dst), n16);
  ctx->launches++;
  return cudaGetLastError();
}

static int tu_buf(vvcb_ctx* ctx, TuSlot i, size_t bytes)
{
  if (bytes > ctx->capTu[i]) {
    cudaFree(ctx->dTu[i]); ctx->dTu[i] = nullptr; ctx->capTu[i] = 0;
    CK(cudaMalloc(&ctx->dTu[i], bytes));
    ctx->capTu[i] = bytes;
  }
  return VVCB_OK;
}

// The counting sort of the dependent quantiser's jobs by first test position buys warp efficiency for sweeps (eight TUs per warp walk
// scans of equal length); a walk's batch of a few dozen candidates is latency bound, skips its three launches and runs one TU per warp.
constexpr int kDqSortAbove = 2048;

static int dq_grid(const vvcb_ctx* ctx, int nDq)
{
  const int g = nDq <= kDqSortAbove ? (nDq + kDqThreads / 32 - 1) / (kDqThreads / 32) : (nDq + kDqGroups - 1) / kDqGroups;
  return std::min(g, ctx->numSms * 4);
}

// Quantiser scratch of one call whose batches hold `samples` samples, nRates price sets and nDq[0..steps) dependent-quantiser jobs:
// pass 0's coefficients, the derived rate tables, per-group context memory + trellis, the first-position / sort lists.  Sized once per
// call, before its first batch: a buffer that grew between two batches would be freed under the previous one's kernels.
static int quant_scratch(vvcb_ctx* ctx, size_t samples, int nRates, const int* nDq, int steps)
{
  int maxDq = 0, maxGrid = 0;                                       // the grid is not monotonic in the job count (sparse, kDqSortAbove)
  for (int k = 0; k < steps; k++) { maxDq = std::max(maxDq, nDq[k]); maxGrid = std::max(maxGrid, dq_grid(ctx, nDq[k])); }
  int rc;
  if ((rc = tu_buf(ctx, kDqCoeff, samples * sizeof(int32_t)))) return rc;
  if (!maxDq) return VVCB_OK;
  if ((rc = tu_buf(ctx, kDqTabs, (size_t)nRates * sizeof(DqRateTab)))) return rc;
  if ((rc = tu_buf(ctx, kDqScratch, (size_t)maxGrid * kDqGroups * kDqSlotBytes))) return rc;
  return tu_buf(ctx, kDqLists, ((size_t)maxDq * 3 + kDqBins) * sizeof(int));
}

// job indices of bySize[log2w + log2h - 4], largest TU first
static std::vector<int> largest_first(const std::vector<int> (&bySize)[9])
{
  std::vector<int> out;
  for (int c = 8; c >= 0; c--) out.insert(out.end(), bySize[c].begin(), bySize[c].end());
  return out;
}

// Host work lists of one TU batch over the jobs i < n with part(i):
// - team: the job list of tu_eval_kernel, the nSmall blocks of up to 256 samples (one warp each) first, then the larger ones;
// - dq: the dependent quantiser's jobs (sorted on the device by scan length once the coefficients exist);
// - ts: the transform-skip RDOQ jobs, largest block first (one thread per block: equal chain lengths per warp);
// - rate: the VVCB_TU_RATE jobs, whose residual bits are wanted, largest TU first.
struct TuLists { std::vector<int> team, dq, ts, rate; int nSmall; };

template <class Part> static TuLists tu_lists(const vvcb_tu_job* jobs, int n, Part part)
{
  TuLists L;
  L.team.reserve(n); L.dq.reserve(n);
  std::vector<int> large, tsBySize[9], rateBySize[9];
  for (int i = 0; i < n; i++) {
    if (!part(i)) continue;
    const vvcb_tu_job& j = jobs[i];
    const int c = j.log2w + j.log2h - 4;
    const bool q = (j.flags & VVCB_TU_QUANT) != 0;
    (c <= 4 ? L.team : large).push_back(i);
    if (q && (j.flags & VVCB_TU_DEPQUANT)) L.dq.push_back(i);
    else if (q && (j.flags & VVCB_TU_RDOQ_TS)) tsBySize[c].push_back(i);
    if (q && (j.flags & VVCB_TU_RATE)) rateBySize[c].push_back(i);
  }
  L.nSmall = (int)L.team.size();
  L.team.insert(L.team.end(), large.rbegin(), large.rend());
  L.ts = largest_first(tsBySize);
  L.rate = largest_first(rateBySize);
  return L;
}

// Device pointers of one TU batch (counts: its TuLists).  The quantiser scratch comes from quant_scratch.
struct TuChain {
  const vvcb_tu_job* jobs;
  const uint8_t* trPair;                                            // optional explicit transform pair per job (TuParams)
  const int *team, *dq, *ts, *rate;                                 // the TuLists
  const int16_t *resi, *pred;
  int32_t* coeff; int32_t* level; int16_t* reco; int32_t* deq; vvcb_tu_result* results;   // coeff, reco optional
  vvcb_dq_rates* rates; int nRates;                                 // quantiser prices
  const vvcb_ctx_states* priceFrom;                                 // optional: rates_from_states_kernel fills `rates` from these models first
  const vvcb_ctx_states* states; vvcb_ctx_states* statesOut;        // rate_kernel's models; statesOut optional
};

// Launches one TU batch: tu_eval_kernel pass 0 in its two team sizes, the dependent quantiser and / or transform-skip RDOQ, pass 1 for
// the jobs they quantised, rate_kernel.  ev (optional): ev[1..4] are recorded after pass 0, the quantisers, pass 1 and rate_kernel.
static int run_tu_chain(vvcb_ctx* ctx, const TuChain& c, const TuLists& L, const cudaEvent_t* ev)
{
  const int nSmall = L.nSmall, nLarge = (int)L.team.size() - nSmall, nDq = (int)L.dq.size(), nTs = (int)L.ts.size(), nRate = (int)L.rate.size();
  TuParams P;
  P.jobs = c.jobs; P.list = nullptr; P.n = 0; P.resi = c.resi; P.pred = c.pred; P.coeff = c.coeff; P.level = c.level; P.reco = c.reco;
  P.results = c.results; P.orig = ctx->bOrig; P.stride = ctx->stride; P.bd = ctx->bd; P.rom = ctx->dTrRom;
  P.dqCoeff = static_cast<int32_t*>(ctx->dTu[kDqCoeff]); P.dqDeq = c.deq; P.phase = 0; P.trPair = c.trPair;
  auto launch_tu = [&](TuParams Q) {
    if (nSmall) { Q.list = c.team; Q.n = nSmall; tu_eval_kernel<32><<<std::min((nSmall + 3) / 4, ctx->numSms * 8), kTuThreads, 0, ctx->stream>>>(Q); ctx->launches++; }
    if (nLarge) { Q.list = c.team + nSmall; Q.n = nLarge; tu_eval_kernel<128><<<std::min(nLarge, ctx->numSms * 8), kTuThreads, 0, ctx->stream>>>(Q); ctx->launches++; }
  };
  launch_tu(P);
  if (ev) CK(cudaEventRecord(ev[1], ctx->stream));
  // transform-skip RDOQ and dependent quantisation work on disjoint jobs: the former runs on a side stream next to the latter
  const bool tsAside = nTs && nDq;
  if (tsAside) {
    CK(cudaEventRecord(ctx->evPlan, ctx->stream));
    CK(cudaStreamWaitEvent(ctx->sKind[0], ctx->evPlan, 0));
  }
  if (nDq) {
    if (c.priceFrom) {
      const long long nPrice = (long long)c.nRates * kDqRateModels;
      rates_from_states_kernel<<<(unsigned)((nPrice + 127) / 128), 128, 0, ctx->stream>>>(c.priceFrom, c.nRates, ctx->dRateRom, c.rates);
      ctx->launches++;
    }
    dq_rate_kernel<<<c.nRates, 32, 0, ctx->stream>>>(c.rates, c.nRates, static_cast<DqRateTab*>(ctx->dTu[kDqTabs]));
    int* firstRaw = static_cast<int*>(ctx->dTu[kDqLists]);
    int* orderSorted = firstRaw + nDq;
    int* firstSorted = firstRaw + 2 * nDq;
    dq_first_kernel<<<std::min((nDq + kDqGroups - 1) / kDqGroups, ctx->numSms * 8), kDqThreads, 0, ctx->stream>>>(c.jobs, c.dq, nDq, P.dqCoeff, ctx->dDqRom, ctx->bd, firstRaw);
    const bool sortJobs = nDq > kDqSortAbove;
    if (sortJobs) {
      int* binCount = firstRaw + 3 * (size_t)nDq;
      const int sortGrid = (nDq + kDqSortPerBlock - 1) / kDqSortPerBlock;
      CK(cudaMemsetAsync(binCount, 0, kDqBins * sizeof(int), ctx->stream));
      dq_hist_kernel<<<sortGrid, kDqSortThreads, 0, ctx->stream>>>(firstRaw, nDq, binCount);
      dq_scan_kernel<<<1, 32, 0, ctx->stream>>>(binCount);
      dq_scatter_kernel<<<sortGrid, kDqSortThreads, 0, ctx->stream>>>(c.dq, firstRaw, nDq, binCount, orderSorted, firstSorted);
      ctx->launches += 3;
    }
    DqParams D;
    D.jobs = c.jobs; D.order = sortJobs ? orderSorted : c.dq; D.firstPos = sortJobs ? firstSorted : firstRaw; D.n = nDq;
    D.coeff = P.dqCoeff; D.level = c.level; D.deq = c.deq; D.results = c.results;
    D.rates = c.rates; D.tabs = static_cast<const DqRateTab*>(ctx->dTu[kDqTabs]);
    D.rom = ctx->dDqRom; D.scratch = static_cast<uint8_t*>(ctx->dTu[kDqScratch]); D.bd = ctx->bd; D.sparse = !sortJobs;
    dq_kernel<<<dq_grid(ctx, nDq), kDqThreads, 0, ctx->stream>>>(D);
    ctx->launches += 3;
  }
  if (nTs) {
    RdoqParams R;
    R.jobs = c.jobs; R.order = c.ts; R.n = nTs; R.coeff = P.dqCoeff; R.level = c.level;
    R.deq = c.deq; R.results = c.results; R.rates = c.rates;
    R.rom = ctx->dDqRom; R.bd = ctx->bd;
    rdoq_ts_kernel<<<std::min((nTs + kTsWarps - 1) / kTsWarps, 16 * ctx->numSms), kTsThreads, 0, tsAside ? ctx->sKind[0] : ctx->stream>>>(R);
    ctx->launches++;
    if (tsAside) {
      CK(cudaEventRecord(ctx->evKind[0], ctx->sKind[0]));
      CK(cudaStreamWaitEvent(ctx->stream, ctx->evKind[0], 0));
    }
  }
  if (ev) CK(cudaEventRecord(ev[2], ctx->stream));
  if (nDq || nTs) {
    P.phase = 1;
    launch_tu(P);
  }
  if (ev) CK(cudaEventRecord(ev[3], ctx->stream));
  if (nRate) {                                                     // levels are final: price them (CABACWriter::residual_coding on the estimator)
    RateParams R;
    R.jobs = c.jobs; R.order = c.rate; R.n = nRate; R.level = c.level; R.results = c.results;
    R.states = c.states; R.statesOut = c.statesOut; R.rom = ctx->dDqRom; R.rate = ctx->dRateRom; R.depQuant = ctx->depQuant;
    rate_kernel<<<std::min((nRate + kRateWarps - 1) / kRateWarps, 16 * ctx->numSms), kRateThreads, 0, ctx->stream>>>(R);
    ctx->launches++;
  }
  if (ev) CK(cudaEventRecord(ev[4], ctx->stream));
  return VVCB_OK;
}

// Common body of vvcb_tu_eval (residual and prediction come from the host) and vvcb_tu_eval_pred (src != nullptr: both are
// produced on the device by tu_pred_kernel from the frame planes).
static int tu_eval_impl(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int16_t* resi, const int16_t* pred, size_t n_samples,
                        const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates, int32_t* coeff, int32_t* level, int16_t* reco, vvcb_tu_result* results,
                        const vvcb_rmd_visit* visits, int n_visits, const vvcb_tu_src* src, int16_t* pred_out, TuWalk* walk = nullptr)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_tu_eval");
  if (n < 0 || n_rates < 0 || (n > 0 && (!jobs || (!results && !walk) || (!src && !resi) || (src && (!visits || n_visits <= 0)))) || (walk && !src)) {
    snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval: bad argument"); return VVCB_ERR_ARG;
  }
  if (n == 0) return VVCB_OK;
  if (src) {
    if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval_pred: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
    const int rcv = check_visits(ctx, visits, n_visits);
    if (rcv) return rcv;
    const int badSrc = first_bad_index(n, [&](int i) {
      bool ok = src[i].visit < (uint32_t)n_visits && src[i].slot < VVCB_NUM_SLOTS;
      if (ok) {
        const vvcb_rmd_visit& v = visits[src[i].visit];
        const bool mrlAllowed = !(v.flags & VVCB_VISIT_NO_MRL) && (v.y & (ctx->ctu - 1)) != 0;
        const int numMip = (v.flags & VVCB_VISIT_NO_MIP) ? 0 : mip_num_modes(1 << v.log2w, 1 << v.log2h);
        const int slot = src[i].slot;
        ok = (slot < VVCB_SLOT_MRL1 || (slot < VVCB_SLOT_MIP ? mrlAllowed : slot - VVCB_SLOT_MIP < numMip)) &&
             jobs[i].x == v.x && jobs[i].y == v.y && jobs[i].log2w == v.log2w && jobs[i].log2h == v.log2h;
      }
      return ok;
    });
    if (badSrc >= 0) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval_pred: source %d is malformed (visit index, slot not evaluated for the visit, or job geometry differs from the visit)", badSrc); return VVCB_ERR_ARG; }
  }
  const int badJob = first_bad_index(n, [&](int i) {
    const vvcb_tu_job& j = jobs[i];
    const size_t sz = (size_t)1 << (j.log2w + j.log2h);
    const bool q = (j.flags & VVCB_TU_QUANT) != 0;
    const bool dq = q && (j.flags & VVCB_TU_DEPQUANT);
    bool ok = j.log2w >= 2 && j.log2w <= 6 && j.log2h >= 2 && j.log2h <= 6 && j.mts_idx <= 5 && (size_t)j.offset + sz <= n_samples &&
              j.qp_rem >= 0 && j.qp_rem < 6 && j.qp_per >= 0 && 6 * j.qp_per + j.qp_rem <= max_qp(ctx->bd);
    if (j.mts_idx == 1) ok = ok && j.log2w <= 5 && j.log2h <= 5;                 // TU::isTSAllowed, CL/UnitTools.cpp:4524
    if (j.mts_idx > 1)  ok = ok && j.log2w <= 5 && j.log2h <= 5;                 // TU::isMTSAllowed, :4549
    if (q) ok = ok && ctx->bOrig && j.x >= 0 && j.y >= 0 && j.x + (1 << j.log2w) <= ctx->width && j.y + (1 << j.log2h) <= ctx->height;
    if (dq) ok = ok && j.mts_idx != 1 && rates && j.rate_idx < n_rates && j.lfnst_idx <= 2 && lambda_ok(j.lambda);   // CL/DepQuant.cpp:1757: TS goes to RDOQ
    if (j.flags & VVCB_TU_RDOQ_TS) ok = ok && q && !dq && j.mts_idx == 1 && rates && j.rate_idx < n_rates && lambda_ok(j.lambda);
    ok = ok && j.lfnst_idx <= 2 && (j.lfnst_idx == 0 || j.intra_mode < VVCB_NUM_LUMA_MODE);
    if (j.flags & VVCB_TU_RATE) ok = ok && q && states && j.rate_idx < n_rates;
    return ok;
  });
  if (badJob >= 0) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval: job %d is malformed", badJob); return VVCB_ERR_ARG; }
  const bool anyQuant = std::any_of(jobs, jobs + n, [](const vvcb_tu_job& j) { return (j.flags & VVCB_TU_QUANT) != 0; });
  if (anyQuant && !pred && !src) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval: VVCB_TU_QUANT needs the prediction samples"); return VVCB_ERR_ARG; }
  const TuLists L = tu_lists(jobs, n, [](int) { return true; });
  const int nDq = (int)L.dq.size(), nTs = (int)L.ts.size(), nRate = (int)L.rate.size();
  CK(cudaSetDevice(ctx->device));
  int rc;
  const bool wLevel = walk ? walk->wantLevel : level != nullptr, wReco = walk ? walk->wantReco : reco != nullptr, wPred = walk ? walk->wantPred : pred_out != nullptr;
  const bool needLevel = wLevel || nDq || nTs || nRate;
  if ((nDq || nTs) && (rc = quant_scratch(ctx, n_samples, n_rates, &nDq, 1))) return rc;
  if ((rc = tu_buf(ctx, kTuResi, n_samples * sizeof(int16_t)))) return rc;
  if (coeff && (rc = tu_buf(ctx, kTuCoeff, n_samples * sizeof(int32_t)))) return rc;
  // the host inputs in one device arena; walk mode stages them in page-locked memory, moved by one copy kernel
  const size_t ratesBytes = (nDq || nTs) ? (size_t)n_rates * sizeof(vvcb_dq_rates) : 0, statesBytes = nRate ? (size_t)n_rates * sizeof(vvcb_ctx_states) : 0;
  Arena in;
  const size_t iJobs = in.take((size_t)n * sizeof(vvcb_tu_job)), iVis = in.take((size_t)n_visits * sizeof(vvcb_rmd_visit)),
               iSrc = in.take(src ? (size_t)n * sizeof(vvcb_tu_src) : 0), iTeam = in.take((size_t)n * sizeof(int)), iOrder = in.take((size_t)nDq * sizeof(int)),
               iTs = in.take((size_t)nTs * sizeof(int)), iRates = in.take(ratesBytes), iRateOrder = in.take((size_t)nRate * sizeof(int)), iStates = in.take(statesBytes);
  uint8_t* hin = nullptr;
  if (walk) {
    if ((rc = pin_buf(ctx, kPinTuIn, in.size))) return rc;
    hin = static_cast<uint8_t*>(ctx->hPin[kPinTuIn]);
  }
  if ((rc = tu_buf(ctx, kTuIn, in.size))) return rc;
  void* din = ctx->dTu[kTuIn];
  auto put = [&](size_t o, const void* p, size_t bytes) {
    if (!bytes) return cudaSuccess;
    if (walk) { memcpy(hin + o, p, bytes); return cudaSuccess; }
    return cudaMemcpyAsync(at<uint8_t>(din, o), p, bytes, cudaMemcpyHostToDevice, ctx->stream);
  };
  CK(put(iJobs, jobs, (size_t)n * sizeof(vvcb_tu_job)));
  if (src) { CK(put(iVis, visits, (size_t)n_visits * sizeof(vvcb_rmd_visit))); CK(put(iSrc, src, (size_t)n * sizeof(vvcb_tu_src))); }
  CK(put(iTeam, L.team.data(), (size_t)n * sizeof(int)));
  CK(put(iOrder, L.dq.data(), (size_t)nDq * sizeof(int)));
  CK(put(iTs, L.ts.data(), (size_t)nTs * sizeof(int)));
  CK(put(iRates, rates, ratesBytes));
  CK(put(iRateOrder, L.rate.data(), (size_t)nRate * sizeof(int)));
  CK(put(iStates, states, statesBytes));
  if (walk) CK(arena_copy(ctx, hin, din, in.size));
  // the outputs in one device arena: results | prediction | reconstruction | levels, then the dequantised coefficients next to the levels
  Arena out;
  const size_t oRes = out.take((size_t)n * sizeof(vvcb_tu_result)), oPred = out.take(n_samples * sizeof(int16_t)),
               oReco = out.take(wReco ? n_samples * sizeof(int16_t) : 0), oLevel = out.take(needLevel ? n_samples * sizeof(int32_t) : 0);
  const size_t outBytes = wLevel ? out.size : (wReco ? oLevel : (wPred ? oReco : oPred));   // walk mode: what travels back
  const size_t oDeq = out.take((nDq || nTs) ? n_samples * sizeof(int32_t) : 0);
  if ((rc = tu_buf(ctx, kTuOut, out.size))) return rc;
  void* dout = ctx->dTu[kTuOut];
  if (walk) {
    if ((rc = pin_buf(ctx, kPinTuOut, outBytes))) return rc;
    void* hout = ctx->hPin[kPinTuOut];
    walk->results = at<vvcb_tu_result>(hout, oRes); walk->pred = at<int16_t>(hout, oPred);
    walk->reco = at<int16_t>(hout, oReco); walk->level = at<int32_t>(hout, oLevel);
  }
  TuChain c = {};
  c.jobs = at<const vvcb_tu_job>(din, iJobs);
  c.team = at<const int>(din, iTeam); c.dq = at<const int>(din, iOrder); c.ts = at<const int>(din, iTs); c.rate = at<const int>(din, iRateOrder);
  int16_t* dPred = at<int16_t>(dout, oPred);
  c.resi = static_cast<const int16_t*>(ctx->dTu[kTuResi]); c.pred = dPred;
  c.coeff = coeff ? static_cast<int32_t*>(ctx->dTu[kTuCoeff]) : nullptr;
  c.level = needLevel ? at<int32_t>(dout, oLevel) : nullptr; c.reco = wReco ? at<int16_t>(dout, oReco) : nullptr;
  c.deq = (nDq || nTs) ? at<int32_t>(dout, oDeq) : nullptr; c.results = at<vvcb_tu_result>(dout, oRes);
  c.rates = at<vvcb_dq_rates>(din, iRates); c.nRates = n_rates; c.states = at<const vvcb_ctx_states>(din, iStates);
  if (nDq || nTs) CK(cudaMemsetAsync(c.level, 0, oDeq - oLevel + n_samples * sizeof(int32_t), ctx->stream));   // levels and dequantised coefficients
                                                                                                               // the quantisers do not reach stay zero
  const bool tm = ctx->timing != 0;
  if (src) {
    if (tm) CK(cudaEventRecord(ctx->tev[0], ctx->stream));
    TuPredParams Q;
    Q.visits = at<const vvcb_rmd_visit>(din, iVis); Q.src = at<const vvcb_tu_src>(din, iSrc); Q.jobs = c.jobs; Q.n = n;
    Q.pred = dPred; Q.resi = static_cast<int16_t*>(ctx->dTu[kTuResi]);
    Q.orig = ctx->bOrig; Q.reco = ctx->bReco; Q.stride = ctx->stride; Q.bd = ctx->bd; Q.ctu = ctx->ctu; Q.rom = ctx->dRom;
    const int pg = (n + kTuPredWarps - 1) / kTuPredWarps < ctx->numSms * 8 ? (n + kTuPredWarps - 1) / kTuPredWarps : ctx->numSms * 8;
    tu_pred_kernel<<<pg, kTuPredWarps * 32, 0, ctx->stream>>>(Q);
    ctx->launches++;
  } else {
    CK(cudaMemcpyAsync(ctx->dTu[kTuResi], resi, n_samples * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
    if (pred) CK(cudaMemcpyAsync(dPred, pred, n_samples * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
    if (tm) CK(cudaEventRecord(ctx->tev[0], ctx->stream));
  }
  if ((rc = run_tu_chain(ctx, c, L, tm ? ctx->tev : nullptr))) return rc;
  CK(cudaGetLastError());
  if (coeff) CK(cudaMemcpyAsync(coeff, c.coeff, n_samples * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (walk) CK(arena_copy(ctx, dout, ctx->hPin[kPinTuOut], outBytes));
  else {
    if (level) CK(cudaMemcpyAsync(level, c.level, n_samples * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (reco) CK(cudaMemcpyAsync(reco, c.reco, n_samples * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (pred_out) CK(cudaMemcpyAsync(pred_out, dPred, n_samples * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(results, c.results, (size_t)n * sizeof(vvcb_tu_result), cudaMemcpyDeviceToHost, ctx->stream));
  }
  if (ctx->cuSpan) CK(cudaEventRecord(ctx->cev[3], ctx->stream));
  ctx->tuWaitFrom = host_ns();
  CK(ctx_sync(ctx));
  if (tm) {
    for (int i = 0; i < 4; i++) { float ms = 0; CK(cudaEventElapsedTime(&ms, ctx->tev[i], ctx->tev[i + 1])); ctx->tuMs[i] += ms; }
    ctx->tuTimed++;
  }
  return VVCB_OK;
}

extern "C" int vvcb_tu_eval(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int16_t* resi, const int16_t* pred, size_t n_samples,
                            const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                            int32_t* coeff, int32_t* level, int16_t* reco, vvcb_tu_result* results)
{
  return tu_eval_impl(ctx, jobs, n, resi, pred, n_samples, rates, states, n_rates, coeff, level, reco, results, nullptr, 0, nullptr, nullptr);
}

extern "C" int vvcb_tu_eval_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_tu_src* src, const vvcb_tu_job* jobs, int n,
                                 size_t n_samples, const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                                 int32_t* coeff, int32_t* level, int16_t* reco, int16_t* pred_out, vvcb_tu_result* results)
{
  if (ctx && n > 0 && !src) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_tu_eval_pred: bad argument"); return VVCB_ERR_ARG; }
  return tu_eval_impl(ctx, jobs, n, nullptr, nullptr, n_samples, rates, states, n_rates, coeff, level, reco, results, visits, n_visits, src, pred_out);
}

#include "vvcb_expand.inc"

// One round trip per CU of a host walk, for any number of independent CUs (several walkers behind the broker): the reconstruction
// rectangles of all requests travel in one copy and one scatter launch, the rough mode decisions of all requests are one launch_rmd
// batch, the TU candidates of all requests one tu_eval_impl batch (job offsets, visit and snapshot indices are re-based onto
// the merged arrays).  Requests with templates (vvcb_cu_auto) are expanded on the host between the two stages, from the lists the
// first stage has just produced.
extern "C" int vvcb_cu_eval(vvcb_ctx* ctx, vvcb_cu_request* reqs, int n)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && !reqs)) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_cu_eval: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  if (ctx->remote) return vvcbc_cu_eval(ctx->remote, reqs, n, ctx->err, sizeof(ctx->err));
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_cu_eval: no frame (vvcb_frame_begin / vvcb_frame_alloc)"); return VVCB_ERR_STATE; }
  size_t nRects = 0, nRectSamples = 0;
  int nRmd = 0;
  bool anyDetail = false, anyAuto = false;
  for (int i = 0; i < n; i++) {
    const vvcb_cu_request& q = reqs[i];
    bool ok = q.n_rects >= 0 && q.n_jobs >= 0 && q.n_autos >= 0 && (!q.n_rects || (q.rects && q.rect_samples)) && (!(q.want_rmd || q.n_jobs || q.n_autos) || q.visit) &&
              (!q.want_rmd || q.result) && (!q.n_jobs || (q.jobs && q.slots && q.tu_results));
    if (ok && q.n_rects && (!ctx->wReco || ctx->bReco != ctx->wReco)) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_cu_eval: rectangles need a writable frame"); return VVCB_ERR_STATE; }
    for (int k = 0; ok && k < q.n_rects; k++) ok = rect_ok(ctx, q.rects[k], q.n_rect_samples);
    if (ok && (q.n_jobs || q.n_autos)) ok = q.visit->log2w >= 2 && q.visit->log2w <= 6 && q.visit->log2h >= 2 && q.visit->log2h <= 6;
    if (ok && q.n_jobs) {
      const size_t bs = (size_t)1 << (q.visit->log2w + q.visit->log2h);
      for (int k = 0; ok && k < q.n_jobs; k++) {
        const vvcb_tu_job& j = q.jobs[k];
        ok = j.rate_idx == 0 && (size_t)j.offset + bs <= (size_t)q.n_jobs * bs &&
             (!(j.flags & (VVCB_TU_DEPQUANT | VVCB_TU_RDOQ_TS)) || q.rates) && (!(j.flags & VVCB_TU_RATE) || q.states);
      }
    }
    if (ok && q.n_autos) {
      ok = q.want_rmd && q.autos && q.max_auto > 0 && q.n_auto && q.auto_slot && q.auto_tmpl && q.auto_results && q.n_autos <= 32;
      for (int k = 0; ok && k < q.n_autos; k++) {
        const vvcb_cu_auto& a = q.autos[k];
        ok = a.job.x == q.visit->x && a.job.y == q.visit->y && a.job.log2w == q.visit->log2w && a.job.log2h == q.visit->log2h &&
             (!(a.modes & VVCB_AUTO_REGULAR) || q.detail) &&
             (!(a.job.flags & (VVCB_TU_DEPQUANT | VVCB_TU_RDOQ_TS)) || q.rates) && (!(a.job.flags & VVCB_TU_RATE) || q.states);
      }
      anyAuto = anyAuto || ok;
    }
    if (!ok) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_cu_eval: request %d is malformed (pointers, rectangle outside the picture, job offset / snapshot, templates)", i); return VVCB_ERR_ARG; }
    nRects += (size_t)q.n_rects; nRectSamples += q.n_rects ? q.n_rect_samples : 0;
    nRmd += q.want_rmd != 0; anyDetail = anyDetail || (q.want_rmd && q.detail);
  }
  CK(cudaSetDevice(ctx->device));
  int rc;
  uint64_t tPhase = host_ns();
  auto phase = [&](int k) { const uint64_t now = host_ns(); ctx->cuNs[k] += now - tPhase; tPhase = now; };
  ctx->cuSpan = true;
  CK(cudaEventRecord(ctx->cev[0], ctx->stream));
  // ---- inputs of the first stage: rectangles | their samples | visits, one page-locked arena, moved by a copy kernel (see TuWalk) ----
  Arena in;
  const size_t iRects = in.take(nRects * sizeof(vvcb_rect)), iSmp = in.take(nRectSamples * sizeof(int16_t)), iVis = in.take((size_t)nRmd * sizeof(vvcb_rmd_visit));
  vvcb_rmd_result* hRes = nullptr; vvcb_rmd_detail* hDet = nullptr;
  if (in.size) {
    if ((rc = pin_buf(ctx, kPinStageIn, in.size))) return rc;
    if ((rc = tu_buf(ctx, kStageIn, in.size))) return rc;
    void* hin = ctx->hPin[kPinStageIn];
    void* din = ctx->dTu[kStageIn];
    vvcb_rect* hr = at<vvcb_rect>(hin, iRects);
    int16_t* hs = at<int16_t>(hin, iSmp);
    vvcb_rmd_visit* hv = at<vvcb_rmd_visit>(hin, iVis);
    size_t ri = 0, so = 0;
    int vi = 0;
    for (int i = 0; i < n; i++) {
      const vvcb_cu_request& q = reqs[i];
      if (q.want_rmd) hv[vi++] = *q.visit;
      if (!q.n_rects) continue;
      for (int k = 0; k < q.n_rects; k++) { hr[ri] = q.rects[k]; hr[ri].offset += (uint32_t)so; ri++; }
      memcpy(hs + so, q.rect_samples, q.n_rect_samples * sizeof(int16_t));
      so += q.n_rect_samples;
    }
    if (nRmd && (rc = check_visits(ctx, hv, nRmd))) return rc;
    CK(arena_copy(ctx, hin, din, in.size));
    // ---- reconstruction rectangles ----
    if (nRects) {
      reco_scatter_kernel<<<(int)nRects < ctx->numSms * 8 ? (int)nRects : ctx->numSms * 8, 128, 0, ctx->stream>>>(at<const vvcb_rect>(din, iRects), (int)nRects,
                                                                                                          at<const int16_t>(din, iSmp), ctx->wReco, ctx->stride);
      ctx->launches++;
      CK(cudaGetLastError());
    }
    // ---- rough mode decision ----
    if (nRmd) {
      Arena out;
      const size_t oRes = out.take((size_t)nRmd * sizeof(vvcb_rmd_result)), oDet = out.take(anyDetail ? (size_t)nRmd * sizeof(vvcb_rmd_detail) : 0);
      if ((rc = tu_buf(ctx, kStageOut, out.size))) return rc;
      if ((rc = pin_buf(ctx, kPinStageOut, out.size))) return rc;
      void* dout = ctx->dTu[kStageOut];
      void* hout = ctx->hPin[kPinStageOut];
      hRes = at<vvcb_rmd_result>(hout, oRes);
      hDet = anyDetail ? at<vvcb_rmd_detail>(hout, oDet) : nullptr;
      if ((rc = launch_rmd(ctx, at<const vvcb_rmd_visit>(din, iVis), nRmd, at<vvcb_rmd_result>(dout, oRes),
                           anyDetail ? at<vvcb_rmd_detail>(dout, oDet) : nullptr, nullptr, hv))) return rc;
      CK(arena_copy(ctx, dout, hout, out.size));
    }
  }
  if (nRmd) {
    CK(cudaEventRecord(ctx->cev[1], ctx->stream));
    phase(0);
    if (anyAuto) { CK(ctx_sync(ctx)); phase(1); }      // the templates are expanded from these lists
  }
  // ---- TU candidates: the explicit jobs of every request and the expanded templates, as groups of one visit each ----
  struct Group { int req; bool autos; int n; const vvcb_tu_job* jobs; const uint8_t* slots; };
  std::vector<Group> groups;
  std::vector<std::vector<vvcb_tu_job>> autoJobs;
  size_t nJobs = 0, nSamples = 0;
  {
    int vi = 0;
    for (int i = 0; i < n; i++) {
      vvcb_cu_request& q = reqs[i];
      if (q.n_jobs) { groups.push_back(Group{ i, false, q.n_jobs, q.jobs, q.slots }); nJobs += (size_t)q.n_jobs; nSamples += (size_t)q.n_jobs << (q.visit->log2w + q.visit->log2h); }
      if (q.n_autos) {
        autoJobs.emplace_back((size_t)q.max_auto);
        const int cnt = vvcb_expand_autos(*q.visit, hRes[vi], q.detail ? &hDet[vi] : nullptr, q.autos, q.n_autos, q.max_auto, autoJobs.back().data(), q.auto_slot, q.auto_tmpl);
        *q.n_auto = cnt;
        if (cnt) { groups.push_back(Group{ i, true, cnt, autoJobs.back().data(), q.auto_slot }); nJobs += (size_t)cnt; nSamples += (size_t)cnt << (q.visit->log2w + q.visit->log2h); }
      }
      vi += q.want_rmd != 0;
    }
  }
  int32_t* hLevel = nullptr; int16_t* hReco = nullptr; int16_t* hPred = nullptr;
  vvcb_tu_result* tuRes = nullptr;
  if (nJobs) {
    TuWalk walk = {};
    for (const Group& g : groups) {
      const vvcb_cu_request& q = reqs[g.req];
      walk.wantLevel = walk.wantLevel || (g.autos ? q.auto_level : q.level); walk.wantReco = walk.wantReco || (g.autos ? q.auto_reco : q.reco);
      walk.wantPred = walk.wantPred || (g.autos ? q.auto_pred : q.pred);
    }
    const int nGroups = (int)groups.size();
    if (nGroups > 65535) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_cu_eval: more than 65535 TU groups in one call"); return VVCB_ERR_ARG; }
    std::vector<vvcb_rmd_visit> tv(nGroups);
    std::vector<vvcb_dq_rates> rates(nGroups);
    std::vector<vvcb_ctx_states> states(nGroups);
    std::vector<vvcb_tu_job> jobs(nJobs);
    std::vector<vvcb_tu_src> src(nJobs);
    size_t ji = 0, so = 0;
    for (int gi = 0; gi < nGroups; gi++) {
      const Group& g = groups[gi];
      const vvcb_cu_request& q = reqs[g.req];
      tv[gi] = *q.visit;
      if (q.rates) rates[gi] = *q.rates; else memset(&rates[gi], 0, sizeof(vvcb_dq_rates));
      if (q.states) states[gi] = *q.states; else memset(&states[gi], 0, sizeof(vvcb_ctx_states));
      for (int k = 0; k < g.n; k++, ji++) {
        jobs[ji] = g.jobs[k]; jobs[ji].offset += (uint32_t)so; jobs[ji].rate_idx = (uint16_t)gi;
        src[ji].visit = (uint32_t)gi; src[ji].slot = g.slots[k]; src[ji].pad[0] = src[ji].pad[1] = src[ji].pad[2] = 0;
      }
      so += (size_t)g.n << (q.visit->log2w + q.visit->log2h);
    }
    phase(2);
    CK(cudaEventRecord(ctx->cev[2], ctx->stream));
    rc = tu_eval_impl(ctx, jobs.data(), (int)nJobs, nullptr, nullptr, nSamples, rates.data(), states.data(), nGroups, nullptr, nullptr, nullptr, nullptr,
                      tv.data(), nGroups, src.data(), nullptr, &walk);
    tuRes = walk.results; hLevel = walk.level; hReco = walk.reco; hPred = walk.pred;
    ctx->cuSpan = false;
    if (rc) { cudaStreamSynchronize(ctx->stream); return rc; }
    { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->cev[2], ctx->cev[3]) == cudaSuccess) ctx->cuNs[7] += (uint64_t)(ms * 1e6f); }
    { const uint64_t now = host_ns(); ctx->cuNs[3] += ctx->tuWaitFrom - tPhase; ctx->cuNs[4] += now - ctx->tuWaitFrom; tPhase = now; }
  } else { phase(2); CK(ctx_sync(ctx)); phase(4); }
  // ---- hand the outputs back ----
  {
    int vi = 0;
    for (int i = 0; i < n; i++) {
      vvcb_cu_request& q = reqs[i];
      if (q.want_rmd) { *q.result = hRes[vi]; if (q.detail) *q.detail = hDet[vi]; vi++; }
    }
    size_t ji = 0, so = 0;
    for (const Group& g : groups) {
      vvcb_cu_request& q = reqs[g.req];
      const size_t ns = (size_t)g.n << (q.visit->log2w + q.visit->log2h);
      int32_t* lv = g.autos ? q.auto_level : q.level; int16_t* rc16 = g.autos ? q.auto_reco : q.reco; int16_t* pr = g.autos ? q.auto_pred : q.pred;
      if (lv) memcpy(lv, hLevel + so, ns * sizeof(int32_t));
      if (rc16) memcpy(rc16, hReco + so, ns * sizeof(int16_t));
      if (pr) memcpy(pr, hPred + so, ns * sizeof(int16_t));
      memcpy(g.autos ? q.auto_results : q.tu_results, tuRes + ji, (size_t)g.n * sizeof(vvcb_tu_result));
      so += ns; ji += (size_t)g.n;
    }
  }
  phase(5);
  ctx->cuSpan = false;
  if (nRmd) { float ms = 0; if (cudaEventElapsedTime(&ms, ctx->cev[0], ctx->cev[1]) == cudaSuccess) ctx->cuNs[6] += (uint64_t)(ms * 1e6f); }
  ctx->cuCalls++;
  return VVCB_OK;
}

extern "C" int vvcb_cu_eval_phases(const vvcb_ctx* ctx, uint64_t ns[8], uint64_t* calls)
{
  if (!ctx || !ns) return VVCB_ERR_ARG;
  for (int i = 0; i < 8; i++) ns[i] = ctx->cuNs[i];
  if (calls) *calls = ctx->cuCalls;
  return VVCB_OK;
}

// CABACWriter::residual_coding on given levels (HOST int32, dense per job at job.offset): jobs carry geometry, mts_idx, the
// VVCB_TU_TS_ALLOWED / VVCB_TU_MTS_ALLOWED switches and rate_idx; bits[i] = fractional bits (0 for an all-zero block).
extern "C" int vvcb_residual_bits(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int32_t* levels, size_t n_samples,
                                  const vvcb_ctx_states* states, int n_states, uint64_t* bits)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_residual_bits");
  if (n < 0 || (n > 0 && (!jobs || !levels || !states || !bits || n_states <= 0))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_residual_bits: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  const int bad = first_bad_index(n, [&](int i) {
    const vvcb_tu_job& j = jobs[i];
    bool ok = j.log2w >= 2 && j.log2w <= 6 && j.log2h >= 2 && j.log2h <= 6 && j.mts_idx <= 5 && j.rate_idx < n_states &&
              (size_t)j.offset + ((size_t)1 << (j.log2w + j.log2h)) <= n_samples;
    if (j.mts_idx >= 1) ok = ok && j.log2w <= 5 && j.log2h <= 5;
    // levels are 16-bit (entropyCodingMinimum / entropyCodingMaximum with maxLog2TrDynamicRange 15, CL/Quant.cpp)
    if (ok) ok = std::all_of(levels + j.offset, levels + j.offset + ((size_t)1 << (j.log2w + j.log2h)), [](int32_t v) { return v >= -32768 && v <= 32767; });
    return ok;
  });
  if (bad >= 0) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_residual_bits: job %d is malformed (geometry, rate_idx, or a level outside [-32768, 32767])", bad); return VVCB_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  int rc;
  std::vector<int> bySize[9];
  for (int i = 0; i < n; i++) bySize[jobs[i].log2w + jobs[i].log2h - 4].push_back(i);
  const std::vector<int> order = largest_first(bySize);
  Arena in;
  const size_t iJobs = in.take((size_t)n * sizeof(vvcb_tu_job)), iLevel = in.take(n_samples * sizeof(int32_t)), iOrder = in.take((size_t)n * sizeof(int)),
               iStates = in.take((size_t)n_states * sizeof(vvcb_ctx_states));
  if ((rc = tu_buf(ctx, kTuIn, in.size))) return rc;
  if ((rc = tu_buf(ctx, kTuOut, (size_t)n * sizeof(vvcb_tu_result)))) return rc;
  void* din = ctx->dTu[kTuIn];
  CK(cudaMemcpyAsync(at<uint8_t>(din, iJobs), jobs, (size_t)n * sizeof(vvcb_tu_job), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(at<uint8_t>(din, iLevel), levels, n_samples * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(at<uint8_t>(din, iOrder), order.data(), (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemcpyAsync(at<uint8_t>(din, iStates), states, (size_t)n_states * sizeof(vvcb_ctx_states), cudaMemcpyHostToDevice, ctx->stream));
  RateParams R;
  R.jobs = at<const vvcb_tu_job>(din, iJobs); R.order = at<const int>(din, iOrder); R.n = n;
  R.level = at<const int32_t>(din, iLevel); R.results = static_cast<vvcb_tu_result*>(ctx->dTu[kTuOut]);
  R.states = at<const vvcb_ctx_states>(din, iStates); R.rom = ctx->dDqRom; R.rate = ctx->dRateRom; R.depQuant = ctx->depQuant;
  rate_kernel<<<std::min((n + kRateWarps - 1) / kRateWarps, 16 * ctx->numSms), kRateThreads, 0, ctx->stream>>>(R);
  ctx->launches++;
  CK(cudaGetLastError());
  std::vector<vvcb_tu_result> res(n);
  CK(cudaMemcpyAsync(res.data(), R.results, (size_t)n * sizeof(vvcb_tu_result), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < n; i++) bits[i] = res[i].frac_bits;
  return VVCB_OK;
}

extern "C" int vvcb_tu_kernel_times(vvcb_ctx* ctx, float ms[4], int* calls)
{
  if (!ctx || !ms) return VVCB_ERR_ARG;
  for (int i = 0; i < 4; i++) { ms[i] = ctx->tuMs[i]; ctx->tuMs[i] = 0.f; }
  if (calls) *calls = ctx->tuTimed;
  ctx->tuTimed = 0;
  return VVCB_OK;
}

// RdCost::calcRdCost (CL/RdCost.cpp:63-74) with m_DistScale = 32768 / lambda (RdCost::setLambda, :76-79): IEEE double, one multiply and
// one add in the reference's order.  Host logic: the walk adds its own header bits to vvcb_tu_result::frac_bits before calling it.
extern "C" double vvcb_calc_rd_cost(double lambda, uint64_t frac_bits, uint64_t distortion)
{
  const volatile double distScale = double(1 << 15) / lambda;
  const volatile double scaled = distScale * double(distortion);
  return scaled + double(frac_bits);
}

// host logic: CL/TrQuant.cpp:1112-1123
extern "C" void vvcb_mts_preselect(const int32_t* sums, int n, int width, int height, int max_cand, uint8_t* selected)
{
  static const double facBB[5] = { 1.2, 1.3, 1.3, 1.4, 1.5 };
  if (n <= 0) return;
  int lg = 0;
  for (int m = width > height ? width : height; m > 1; m >>= 1) lg++;
  const double fac = facBB[lg - 2];
  const double thr = fac * sums[0], thrTS = sums[0];
  int tests = 0;
  for (int i = 0; i < n; i++) {
    const bool t = sums[i] <= (i == 1 ? thrTS : thr) && tests <= max_cand;
    selected[i] = t ? 1 : 0;
    tests += t;
  }
}

// host logic: geometry of an intra sub-partition CU (include/vvc_intra_b200.h; CL/UnitTools.cpp:426-460, :4334-4355,
// CL/UnitPartitioner.cpp:978, CL/IntraPrediction.cpp:1092-1203, CL/TrQuant.cpp:752-783).  Everything follows from the two log2
// sizes: a block keeps at least 16 samples, so along the split the CU is cut in four unless that would leave fewer (then in blocks
// of 16 / other-side samples: two of them for 4x8 and 8x4).
extern "C" int vvcb_isp_plan(int cu_w, int cu_h, int isp_mode, int max_tb_size, int use_mts, vvcb_isp_part* parts)
{
  auto lg2 = [](int v) { int l = 0; if (v > 64) return -1; while ((1 << l) < v) l++; return (1 << l) == v ? l : -1; };
  const int lw = lg2(cu_w), lh = lg2(cu_h);
  if (!parts || lw < 2 || lw > 6 || lh < 2 || lh > 6 || (isp_mode != VVCB_ISP_HOR && isp_mode != VVCB_ISP_VER)) return VVCB_ERR_ARG;
  if (lw + lh <= 4 || cu_w > max_tb_size || cu_h > max_tb_size) return 0;
  const bool hor = isp_mode == VVCB_ISP_HOR;
  const int split = hor ? cu_h : cu_w, other = hor ? cu_w : cu_h;
  const int floorSize = other < 16 ? 16 / other : 1;                 // smallest block extent that still holds 16 samples
  const int size = (split >> 2) < floorSize ? floorSize : (split >> 2);
  const int n = split / size;
  // 4xN and 8xN (N > 4) cut vertically: blocks 1 or 2 samples wide, predicted four columns at a time
  const bool wideRegions = !hor && (cu_w == 4 || (cu_w == 8 && cu_h > 4));
  for (int i = 0; i < n; i++) {
    vvcb_isp_part& p = parts[i];
    p.x = int16_t(hor ? 0 : i * size); p.y = int16_t(hor ? i * size : 0);
    p.w = int16_t(hor ? cu_w : size);  p.h = int16_t(hor ? size : cu_h);
    p.pred_x = p.x; p.pred_y = p.y; p.pred_w = p.w; p.pred_h = p.h; p.predicts = 1;
    if (wideRegions && size < 4) {
      p.pred_x = int16_t(p.x & ~3); p.pred_w = 4;
      p.predicts = (p.x & 3) == 0;
    }
    p.top_ref_len = int16_t(cu_w + p.pred_w); p.left_ref_len = int16_t(cu_h + p.pred_h);
    p.fetch_top_len = p.fetch_left_len = 0;
    if (i == 0) {
      p.fetch_top_len  = int16_t(hor ? cu_w + p.pred_w : 2 * cu_w);
      p.fetch_left_len = int16_t(hor ? 2 * cu_h : cu_h + p.pred_h);
    }
    p.tr_hor = uint8_t(use_mts && p.w >= 4 && p.w <= 16 ? VVCB_TR_DST7 : VVCB_TR_DCT2);
    p.tr_ver = uint8_t(use_mts && p.h >= 4 && p.h <= 16 ? VVCB_TR_DST7 : VVCB_TR_DCT2);
    p.last = i == n - 1;
  }
  return n;
}

// host logic: prediction parameters of one mode for a prediction region of an ISP CU (include/vvc_intra_b200.h)
extern "C" int vvcb_isp_mode_param(int cu_w, int cu_h, int pred_w, int pred_h, int mode, vvcb_isp_mode* out)
{
  auto pow2 = [](int v, int lo) { return v >= lo && v <= 64 && (v & (v - 1)) == 0; };
  if (!out || !pow2(cu_w, 4) || !pow2(cu_h, 4) || !pow2(pred_w, 1) || !pow2(pred_h, 1) || pred_w > cu_w || pred_h > cu_h || mode < 0 || mode > 66) return VVCB_ERR_ARG;
  const ModeParam p = make_mode_param_isp(cu_w, cu_h, pred_w, pred_h, mode);
  out->angle = p.angle; out->inv_angle = p.inv_angle; out->is_ver = p.is_ver; out->pdpc = p.pdpc; out->ang_scale = p.ang_scale; out->pad = 0;
  return VVCB_OK;
}

// ISP candidates (include/vvc_intra_b200.h): up to four steps, one per block index k, over the TU kernels; the blocks of every candidate
// that has a block k run in step k: isp_pred_kernel (lines from block k-1's reconstruction, prediction, residual, cbf of block k-1 and
// cbfDeltaBits of block k), tu_eval_kernel pass 0, the quantiser (the dependent one priced by rates_from_states_kernel from the models the
// previous block left), pass 1 (reconstruction into the candidate's buffer), rate_kernel adapting the candidate's carried models in place.
// A fifth isp_pred_kernel pass codes the cbf of the last block of four-block candidates.
// One chunk of at most kIspChunk candidates (their TU jobs name the carried snapshots with the 16-bit rate_idx); base: index of the
// chunk's first job in the caller's batch.  checkOnly: validate, launch nothing.
constexpr int kIspChunk = 65536;
static int isp_eval_chunk(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_isp_job* jobs, int n, int base,
                          const vvcb_ctx_states* states, int n_states, size_t n_samples,
                          int32_t* level, int16_t* reco, int16_t* pred, vvcb_isp_result* results, bool checkOnly)
{
  const unsigned kFlags = VVCB_TU_QUANT | VVCB_TU_DEPQUANT | VVCB_TU_RATE;
  std::vector<IspCand> cands(n);
  std::vector<vvcb_tu_job> tj((size_t)4 * n);
  std::vector<uint8_t> trPair((size_t)4 * n, 0);
  std::vector<IspState> ist(n);
  std::vector<vvcb_ctx_states> cst(n);
  size_t cs = 0;                                   // the chunk's own samples: candidates are packed densely on the device, whatever the caller's offsets
  for (int i = 0; i < n; i++) {
    const vvcb_isp_job& j = jobs[i];
    auto bad = [&](const char* why) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_isp_eval: job %d: %s", base + i, why); return VVCB_ERR_ARG; };
    if (j.visit >= (uint32_t)n_visits) return bad("visit index out of range");
    const vvcb_rmd_visit& v = visits[j.visit];
    const int cuW = 1 << v.log2w, cuH = 1 << v.log2h;
    vvcb_isp_part parts[VVCB_ISP_MAX_PARTS];
    const int np = vvcb_isp_plan(cuW, cuH, j.isp_mode, j.max_tb_size, j.use_mts, parts);
    if (np <= 0) return bad("the CU may not use this split (vvcb_isp_plan)");
    if (parts[0].w < 4 || parts[0].h < 4) return bad("blocks narrower than 4 samples are not evaluated");
    // all-or-nothing availability: the fresh fetch of isp_pred_kernel equals the reference's shifted lines only then
    if ((v.n_left != 0 && v.n_left != cuH / 4) || (v.n_above != 0 && v.n_above != cuW / 4) || (!v.n_left && v.n_below_left) || (!v.n_above && v.n_above_right))
      return bad("left / above availability is not all or nothing");
    if (j.mode >= VVCB_NUM_LUMA_MODE) return bad("mode above 66");
    if (j.lfnst_idx != 0) return bad("LFNST with ISP is not evaluated");
    if ((j.flags & ~kFlags) || !(j.flags & VVCB_TU_QUANT)) return bad("flags: VVCB_TU_QUANT [| VVCB_TU_DEPQUANT] [| VVCB_TU_RATE] only");
    if (j.qp_rem < 0 || j.qp_rem >= 6 || j.qp_per < 0 || 6 * j.qp_per + j.qp_rem > max_qp(ctx->bd)) return bad("qp_per / qp_rem out of range");
    const bool dq = (j.flags & VVCB_TU_DEPQUANT) != 0, carried = dq || (j.flags & VVCB_TU_RATE);
    if (carried && (!states || j.rate_idx >= n_states)) return bad("rate_idx does not name a context snapshot");
    if (dq && !lambda_ok(j.lambda)) return bad("dependent quantisation needs a finite lambda > 0");
    if ((size_t)j.offset + (size_t)cuW * cuH > n_samples) return bad("outputs outside n_samples");
    IspCand& c = cands[i];
    c.x = v.x; c.y = v.y; c.cuW = (int16_t)cuW; c.cuH = (int16_t)cuH; c.bw = parts[0].w; c.bh = parts[0].h;
    c.topLen = parts[0].top_ref_len; c.leftLen = parts[0].left_ref_len;
    c.hor = j.isp_mode == VVCB_ISP_HOR; c.nParts = (uint8_t)np; c.availAl = v.avail_al; c.nAbove = v.n_above; c.nAboveRight = v.n_above_right;
    c.nLeft = v.n_left; c.nBelowLeft = v.n_below_left; c.mode = j.mode; c.offset = (uint32_t)cs;
    c.p = make_mode_param_isp(cuW, cuH, parts[0].pred_w, parts[0].pred_h, j.mode);
    memset(&ist[i], 0, sizeof(IspState));
    ist[i].ctx[0] = j.cbf[0]; ist[i].ctx[1] = j.cbf[1];
    if (carried) cst[i] = states[j.rate_idx]; else memset(&cst[i], 0, sizeof(vvcb_ctx_states));
    for (int k = 0; k < np; k++) {
      vvcb_tu_job& t = tj[(size_t)k * n + i];
      memset(&t, 0, sizeof(t));
      t.x = (int16_t)(v.x + parts[k].x); t.y = (int16_t)(v.y + parts[k].y);
      t.log2w = (uint8_t)vlog2(parts[k].w); t.log2h = (uint8_t)vlog2(parts[k].h);
      t.mts_idx = 0;
      t.flags = (uint8_t)(j.flags | (carried ? VVCB_TU_RATE : 0));   // rate_kernel adapts the carried models of DEPQUANT candidates too
      t.qp_per = j.qp_per; t.qp_rem = j.qp_rem;
      t.offset = (uint32_t)(cs + (size_t)k * parts[k].w * parts[k].h);
      t.rate_idx = (uint16_t)i;                        // the candidate's own carried snapshot
      t.lambda = j.lambda;
      trPair[(size_t)k * n + i] = (uint8_t)(parts[k].tr_hor | parts[k].tr_ver << 2);
    }
    cs += (size_t)cuW * cuH;
  }
  if (checkOnly) return VVCB_OK;
  // per-step work lists (all host-known: the values change, the shapes do not)
  std::vector<int> predList[5];
  TuLists L[4];
  for (int k = 0; k <= 4; k++)
    for (int i = 0; i < n; i++) if (cands[i].nParts > k || (k > 0 && cands[i].nParts == k)) predList[k].push_back(i);
  for (int k = 0; k < 4; k++) L[k] = tu_lists(&tj[(size_t)k * n], n, [&](int i) { return cands[i].nParts > k; });
  // one input arena in page-locked memory: candidates, TU jobs, transform pairs, cbf state, carried models, lists
  Arena in;
  const size_t iCand = in.take((size_t)n * sizeof(IspCand)), iJobs = in.take(tj.size() * sizeof(vvcb_tu_job)), iTr = in.take(trPair.size()),
               iState = in.take((size_t)n * sizeof(IspState)), iCst = in.take((size_t)n * sizeof(vvcb_ctx_states));
  size_t iPred[5], iTeam[4], iDq[4], iRate[4];
  for (int k = 0; k <= 4; k++) iPred[k] = in.take(predList[k].size() * sizeof(int));
  for (int k = 0; k < 4; k++) { iTeam[k] = in.take(L[k].team.size() * sizeof(int)); iDq[k] = in.take(L[k].dq.size() * sizeof(int)); iRate[k] = in.take(L[k].rate.size() * sizeof(int)); }
  int rc;
  if ((rc = pin_buf(ctx, kPinStageIn, in.size))) return rc;
  void* hin = ctx->hPin[kPinStageIn];
  memcpy(at<IspCand>(hin, iCand), cands.data(), (size_t)n * sizeof(IspCand));
  memcpy(at<vvcb_tu_job>(hin, iJobs), tj.data(), tj.size() * sizeof(vvcb_tu_job));
  memcpy(at<uint8_t>(hin, iTr), trPair.data(), trPair.size());
  memcpy(at<IspState>(hin, iState), ist.data(), (size_t)n * sizeof(IspState));
  memcpy(at<vvcb_ctx_states>(hin, iCst), cst.data(), (size_t)n * sizeof(vvcb_ctx_states));
  auto put = [&](size_t o, const std::vector<int>& v) { if (!v.empty()) memcpy(at<int>(hin, o), v.data(), v.size() * sizeof(int)); };
  for (int k = 0; k <= 4; k++) put(iPred[k], predList[k]);
  for (int k = 0; k < 4; k++) { put(iTeam[k], L[k].team); put(iDq[k], L[k].dq); put(iRate[k], L[k].rate); }
  // work arena: per-step TU results, prediction, residual, reconstruction, levels, dequantised coefficients, derived prices
  Arena work;
  const size_t oRes = work.take((size_t)4 * n * sizeof(vvcb_tu_result)), oPred = work.take(cs * sizeof(int16_t)), oResi = work.take(cs * sizeof(int16_t)),
               oReco = work.take(cs * sizeof(int16_t)), oLevel = work.take(cs * sizeof(int32_t)), oDeq = work.take(cs * sizeof(int32_t)),
               oRates = work.take((size_t)n * sizeof(vvcb_dq_rates));
  const int nDq[4] = { (int)L[0].dq.size(), (int)L[1].dq.size(), (int)L[2].dq.size(), (int)L[3].dq.size() };
  CK(cudaSetDevice(ctx->device));
  if ((rc = tu_buf(ctx, kStageIn, in.size))) return rc;
  if ((rc = tu_buf(ctx, kStageOut, work.size))) return rc;
  if ((rc = quant_scratch(ctx, cs, n, nDq, 4))) return rc;
  void* din = ctx->dTu[kStageIn];
  void* dw = ctx->dTu[kStageOut];
  CK(cudaMemcpyAsync(din, hin, in.size, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaMemsetAsync(at<uint8_t>(dw, oLevel), 0, oRates - oLevel, ctx->stream));        // levels / dequantised coefficients the quantisers do not reach stay zero
  const IspCand* dCand = at<const IspCand>(din, iCand);
  vvcb_tu_job* dJobs = at<vvcb_tu_job>(din, iJobs);
  IspState* dState = at<IspState>(din, iState);
  vvcb_ctx_states* dCst = at<vvcb_ctx_states>(din, iCst);
  vvcb_tu_result* dRes = at<vvcb_tu_result>(dw, oRes);
  int16_t* dPred = at<int16_t>(dw, oPred); int16_t* dResi = at<int16_t>(dw, oResi);
  int16_t* dReco = at<int16_t>(dw, oReco); int32_t* dLevel = at<int32_t>(dw, oLevel);
  const bool tm = ctx->timing != 0;
  struct Events {                                    // per-stage timing of the steps (vvcb_tu_kernel_times); destroyed on every exit
    cudaEvent_t e[5 * 4] = {};
    ~Events() { for (auto& x : e) if (x) cudaEventDestroy(x); }
  } tev;
  cudaEvent_t* ev = tev.e;
  if (tm) for (auto& e : tev.e) CK(cudaEventCreate(&e));
  for (int k = 0; k <= 4; k++) {
    if (tm && k < 4) CK(cudaEventRecord(ev[5 * k], ctx->stream));
    if (!predList[k].empty()) {
      IspPredParams Q;
      Q.cands = dCand; Q.list = at<const int>(din, iPred[k]); Q.n = (int)predList[k].size(); Q.k = k;
      Q.jobs = dJobs + (size_t)(k < 4 ? k : 3) * n; Q.prev = dRes + (size_t)(k > 0 ? k - 1 : 0) * n; Q.state = dState;
      Q.pred = dPred; Q.resi = dResi; Q.cuReco = dReco; Q.orig = ctx->bOrig; Q.reco = ctx->bReco; Q.stride = ctx->stride; Q.bd = ctx->bd;
      Q.rom = ctx->dRom; Q.frac = ctx->dRateRom->binFracBits;
      const int g = std::min((Q.n + kIspPredWarps - 1) / kIspPredWarps, ctx->numSms * 8);
      isp_pred_kernel<<<g, kIspPredWarps * 32, 0, ctx->stream>>>(Q);
      ctx->launches++;
    }
    if (k == 4 || L[k].team.empty()) continue;
    TuChain c = {};
    c.jobs = dJobs + (size_t)k * n; c.trPair = at<const uint8_t>(din, iTr) + (size_t)k * n;
    c.team = at<const int>(din, iTeam[k]); c.dq = at<const int>(din, iDq[k]); c.rate = at<const int>(din, iRate[k]);
    c.resi = dResi; c.pred = dPred; c.level = dLevel; c.reco = dReco; c.deq = at<int32_t>(dw, oDeq); c.results = dRes + (size_t)k * n;
    c.rates = at<vvcb_dq_rates>(dw, oRates); c.nRates = n; c.priceFrom = dCst;
    c.states = dCst; c.statesOut = dCst;                             // the block's models adapted in place for the next block
    if ((rc = run_tu_chain(ctx, c, L[k], tm ? ev + 5 * k : nullptr))) return rc;
  }
  CK(cudaGetLastError());
  // page-locked output staging: per-step results, cbf state, then the wanted sample outputs of the chunk's densely packed candidates
  Arena out;
  const size_t hRes = out.take((size_t)4 * n * sizeof(vvcb_tu_result)), hSt = out.take((size_t)n * sizeof(IspState)),
               hLv = out.take(level ? cs * sizeof(int32_t) : 0), hRc = out.take(reco ? cs * sizeof(int16_t) : 0), hPr = out.take(pred ? cs * sizeof(int16_t) : 0);
  if ((rc = pin_buf(ctx, kPinStageOut, out.size))) return rc;
  void* hout = ctx->hPin[kPinStageOut];
  CK(cudaMemcpyAsync(at<uint8_t>(hout, hRes), dRes, (size_t)4 * n * sizeof(vvcb_tu_result), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaMemcpyAsync(at<uint8_t>(hout, hSt), dState, (size_t)n * sizeof(IspState), cudaMemcpyDeviceToHost, ctx->stream));
  if (level) CK(cudaMemcpyAsync(at<uint8_t>(hout, hLv), dLevel, cs * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (reco) CK(cudaMemcpyAsync(at<uint8_t>(hout, hRc), dReco, cs * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
  if (pred) CK(cudaMemcpyAsync(at<uint8_t>(hout, hPr), dPred, cs * sizeof(int16_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(ctx_sync(ctx));
  const vvcb_tu_result* res = at<const vvcb_tu_result>(hout, hRes);
  memcpy(ist.data(), at<IspState>(hout, hSt), (size_t)n * sizeof(IspState));
  for (int i = 0; i < n; i++) {                      // each candidate's samples to the caller's offset
    const size_t from = cands[i].offset, to = jobs[i].offset, m = (size_t)cands[i].cuW * cands[i].cuH;
    if (level) memcpy(level + to, at<const int32_t>(hout, hLv) + from, m * sizeof(int32_t));
    if (reco) memcpy(reco + to, at<const int16_t>(hout, hRc) + from, m * sizeof(int16_t));
    if (pred) memcpy(pred + to, at<const int16_t>(hout, hPr) + from, m * sizeof(int16_t));
  }
  if (tm) {
    for (int k = 0; k < 4; k++) {
      if (L[k].team.empty()) continue;
      for (int i = 0; i < 4; i++) { float ms = 0; CK(cudaEventElapsedTime(&ms, ev[5 * k + i], ev[5 * k + i + 1])); ctx->tuMs[i] += ms; }
    }
    ctx->tuTimed++;
  }
  for (int i = 0; i < n; i++) {
    vvcb_isp_result& r = results[i];
    memset(&r, 0, sizeof(r));
    const int np = cands[i].nParts;
    r.n_parts = (uint8_t)np;
    for (int k = 0; k < np; k++) {
      r.part[k] = res[(size_t)k * n + i];
      if (!(jobs[i].flags & VVCB_TU_RATE)) r.part[k].frac_bits = 0;
      r.cbf_bits[k] = ist[i].cbfBits[k];
      r.cbf[k] = ist[i].cbf[k];
    }
    r.discarded = !ist[i].anyCbf;                                    // the last cbf was inferred (1) but that block has no level either
  }
  return VVCB_OK;
}

extern "C" int vvcb_isp_eval(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_isp_job* jobs, int n,
                             const vvcb_ctx_states* states, int n_states, size_t n_samples,
                             int32_t* level, int16_t* reco, int16_t* pred, vvcb_isp_result* results)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_isp_eval");
  if (n < 0 || n_states < 0 || (n > 0 && (!jobs || !results || !visits || n_visits <= 0))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_isp_eval: bad argument"); return VVCB_ERR_ARG; }
  if (n == 0) return VVCB_OK;
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_isp_eval: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  const int rcv = check_visits(ctx, visits, n_visits);
  if (rcv) return rcv;
  for (int pass = 0; pass < 2; pass++)                               // every job is validated before anything runs
    for (int b = 0; b < n; b += kIspChunk) {
      const int rc = isp_eval_chunk(ctx, visits, n_visits, jobs + b, std::min(kIspChunk, n - b), b, states, n_states, n_samples,
                                    level, reco, pred, results + b, pass == 0);
      if (rc) return rc;
    }
  return VVCB_OK;
}

static int feat_buf(vvcb_ctx* ctx, int i, size_t bytes)
{
  if (bytes > ctx->capFeat[i]) {
    cudaFree(ctx->dFeat[i]); ctx->dFeat[i] = nullptr; ctx->capFeat[i] = 0;
    CK(cudaMalloc(&ctx->dFeat[i], bytes));
    ctx->capFeat[i] = bytes;
  }
  return VVCB_OK;
}

extern "C" int vvcb_ctu_hads_islice(vvcb_ctx* ctx, int32_t* out, int n_ctus)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_ctu_hads_islice");
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_ctu_hads_islice: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  const int perRow = (ctx->width + ctx->ctu - 1) / ctx->ctu, rows = (ctx->height + ctx->ctu - 1) / ctx->ctu;
  if (!out || n_ctus != perRow * rows) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_ctu_hads_islice: the frame has %d CTUs", perRow * rows); return VVCB_ERR_ARG; }
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = feat_buf(ctx, 0, (size_t)n_ctus * sizeof(int32_t)))) return rc;
  int32_t* d = static_cast<int32_t*>(ctx->dFeat[0]);
  CK(cudaMemsetAsync(d, 0, (size_t)n_ctus * sizeof(int32_t), ctx->stream));
  const int blocks = (ctx->width >> 3) * (ctx->height >> 3);
  if (blocks > 0) {
    ctu_hads_kernel<<<(blocks + 255) / 256, 256, 0, ctx->stream>>>(ctx->bOrig, ctx->stride, ctx->width, ctx->height, ctx->ctu, perRow, d);
    ctx->launches++;
    CK(cudaGetLastError());
  }
  CK(cudaMemcpyAsync(out, d, (size_t)n_ctus * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

static bool feat_cu_ok(const vvcb_ctx* ctx, const vvcb_feat_cu& c)
{
  return c.w >= 4 && c.h >= 4 && c.w <= kFeatMaxSide && c.h <= kFeatMaxSide && !(c.w & (c.w - 1)) && !(c.h & (c.h - 1)) &&
         c.x >= 0 && c.y >= 0 && c.x + c.w <= ctx->width && c.y + c.h <= ctx->height;
}

extern "C" int vvcb_features_eval(vvcb_ctx* ctx, const vvcb_feat_job* jobs, int n, vvcb_feat_result* results)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_features_eval");
  if (n < 0 || (n > 0 && (!jobs || !results))) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_features_eval: bad argument"); return VVCB_ERR_ARG; }
  if (!ctx->bOrig) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_features_eval: vvcb_frame_begin has not been called"); return VVCB_ERR_STATE; }
  if (n == 0) return VVCB_OK;
  for (int i = 0; i < n; i++) {
    bool ok = feat_cu_ok(ctx, jobs[i].cu) && jobs[i].n_neighbours <= 5;
    for (int k = 0; ok && k < jobs[i].n_neighbours; k++) ok = feat_cu_ok(ctx, jobs[i].nb[k]);
    if (!ok) { snprintf(ctx->err, sizeof(ctx->err), "vvcb_features_eval: job %d is malformed (sizes are powers of two in 4..64 inside the picture, <= 5 neighbours)", i); return VVCB_ERR_ARG; }
  }
  CK(cudaSetDevice(ctx->device));
  int rc;
  if ((rc = feat_buf(ctx, 0, (size_t)n * sizeof(vvcb_feat_job)))) return rc;
  if ((rc = feat_buf(ctx, 1, (size_t)n * sizeof(vvcb_feat_result)))) return rc;
  CK(cudaMemcpyAsync(ctx->dFeat[0], jobs, (size_t)n * sizeof(vvcb_feat_job), cudaMemcpyHostToDevice, ctx->stream));
  FeatParams P;
  P.jobs = static_cast<const vvcb_feat_job*>(ctx->dFeat[0]); P.n = n; P.results = static_cast<vvcb_feat_result*>(ctx->dFeat[1]);
  P.orig = ctx->bOrig; P.stride = ctx->stride;
  const int grid = n < ctx->numSms * 16 ? n : ctx->numSms * 16;
  features_kernel<<<grid, kFeatThreads, 0, ctx->stream>>>(P);
  ctx->launches++;
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(results, ctx->dFeat[1], (size_t)n * sizeof(vvcb_feat_result), cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}

extern "C" int vvcb_dev_alloc(vvcb_ctx* ctx, size_t bytes, void** out)
{
  if (!ctx || !out) return VVCB_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaMalloc(out, bytes));
  return VVCB_OK;
}
extern "C" int vvcb_dev_free(vvcb_ctx* ctx, void* p)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_dev_free");
  REMOTE_UNAVAILABLE("vvcb_dev_alloc");
  CK(cudaSetDevice(ctx->device));
  CK(cudaFree(p));
  return VVCB_OK;
}
extern "C" int vvcb_host_alloc(vvcb_ctx* ctx, size_t bytes, void** out)
{
  if (!ctx || !out) return VVCB_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaHostAlloc(out, bytes, cudaHostAllocDefault));
  return VVCB_OK;
}
extern "C" int vvcb_host_free(vvcb_ctx* ctx, void* p)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_host_free");
  REMOTE_UNAVAILABLE("vvcb_host_alloc");
  CK(cudaFreeHost(p));
  return VVCB_OK;
}
extern "C" int vvcb_dev_upload(vvcb_ctx* ctx, void* dst, const void* src, size_t bytes)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_dev_upload");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}
extern "C" int vvcb_dev_download(vvcb_ctx* ctx, void* dst, const void* src, size_t bytes)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_dev_download");
  CK(cudaSetDevice(ctx->device));
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}
extern "C" int vvcb_sync(vvcb_ctx* ctx)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_sync");
  CK(cudaSetDevice(ctx->device));
  CK(cudaStreamSynchronize(ctx->stream));
  return VVCB_OK;
}
extern "C" int vvcb_timer_start(vvcb_ctx* ctx)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_timer_start");
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->ev0, ctx->stream));
  return VVCB_OK;
}
extern "C" int vvcb_timer_stop(vvcb_ctx* ctx, float* ms)
{
  if (!ctx || !ms) return VVCB_ERR_ARG;
  CK(cudaSetDevice(ctx->device));
  CK(cudaEventRecord(ctx->ev1, ctx->stream));
  CK(cudaEventSynchronize(ctx->ev1));
  CK(cudaEventElapsedTime(ms, ctx->ev0, ctx->ev1));
  return VVCB_OK;
}
extern "C" int vvcb_measure_int_peak(vvcb_ctx* ctx, double* gops_imad, double* gops_alu, double* gops_mixed)
{
  if (!ctx) return VVCB_ERR_ARG;
  REMOTE_UNAVAILABLE("vvcb_measure_int_peak");
  REMOTE_UNAVAILABLE("vvcb_timer_stop");
  CK(cudaSetDevice(ctx->device));
  const int grid = ctx->numSms * 8, iters = 4096;
  int *dIn = nullptr, *dOut = nullptr;
  CK(cudaMalloc(&dIn, 64 * sizeof(int)));
  CK(cudaMalloc(&dOut, (size_t)grid * 256 * sizeof(int)));
  int hIn[64];
  for (int i = 0; i < 64; i++) hIn[i] = 3 + 2 * i;
  CK(cudaMemcpy(dIn, hIn, sizeof(hIn), cudaMemcpyHostToDevice));
  double* outs[3] = { gops_imad, gops_alu, gops_mixed };
  // lane-operations per thread: KIND 0: 64 IMAD per iteration; KIND 1: 2 ops per statement -> 128; KIND 2: 32 IMAD + 64 ALU
  const double opsPerIter[3] = { 64.0, 128.0, 96.0 };
  for (int kind = 0; kind < 3; kind++) {
    float best = 1e30f;
    for (int rep = 0; rep < 4; rep++) {
      CK(cudaEventRecord(ctx->ev0, ctx->stream));
      if (kind == 0) int_peak_kernel<0><<<grid, 256, 0, ctx->stream>>>(dIn, dOut, iters);
      if (kind == 1) int_peak_kernel<1><<<grid, 256, 0, ctx->stream>>>(dIn, dOut, iters);
      if (kind == 2) int_peak_kernel<2><<<grid, 256, 0, ctx->stream>>>(dIn, dOut, iters);
      CK(cudaEventRecord(ctx->ev1, ctx->stream));
      CK(cudaEventSynchronize(ctx->ev1));
      float ms = 0;
      CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
      if (rep > 0 && ms < best) best = ms;
    }
    if (outs[kind]) *outs[kind] = opsPerIter[kind] * iters * (double)grid * 256.0 / (best * 1e-3) / 1e9;
  }
  cudaFree(dIn); cudaFree(dOut);
  return VVCB_OK;
}
extern "C" uint64_t vvcb_launch_count(const vvcb_ctx* ctx) { return ctx ? ctx->launches : 0; }

// the frame-parallel gather (include/vvc_intra_b200_gather.h): host code only
#include "vvcb_gather.inc"
