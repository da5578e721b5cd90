// TEST INFRASTRUCTURE -- an oracle-backed stand-in for libvvc_intra_b200.so.
//
// Implements the part of the C ABI (include/vvc_intra_b200.h) that the reference-encoder shims (oracle/ref_gpu_shim.cpp,
// oracle/ref_gpu_serve.cpp) and the broker (vvc_intra_b200/csrc/vvcb_broker.inc) use, with the plain-C oracle doing the
// arithmetic.  It exists so that the HOST logic above the ABI -- the substituting shim inside the reference encoder, the
// prefetch cache, the shared-memory broker and its batching -- can be developed and tested in the container that has no GPU
// (tests/test_serve_shim.py, -m "not gpu").  It is never shipped, never on a measured path, and the product library never
// links it: on the GPU box the same binaries load vvc_intra_b200/libvvc_intra_b200.so instead.
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>
#include <map>
#include <mutex>
#include "../../oracle/vvc_oracle.h"
#include "../../include/vvc_intra_b200_broker.h"

struct vvcb_ctx {
  int bd, ctu, depQuant;
  int width, height;
  std::vector<int16_t> origOwn, recoOwn;
  std::vector<int16_t>* origP; std::vector<int16_t>* recoP;   // own planes, or another context's (vvcb_frame_share)
  void* remote;                 // broker client proxy (vvcb_broker.inc)
  char err[512];
};

static char g_createErr[512] = "";
static std::mutex g_oracleMutex;      // the oracle keeps static scratch (single-threaded checker): the broker's worker threads take turns
#define FAIL(code, ...) do { snprintf(ctx->err, sizeof(ctx->err), __VA_ARGS__); return code; } while (0)

#define VVCB_BROKER_IMPL_FAKE 1
#include "../../vvc_intra_b200/csrc/vvcb_broker.inc"
#include "../../vvc_intra_b200/csrc/vvcb_expand.inc"

extern "C" {

int vvcb_device_count(void) { return 1; }
uint64_t vvcb_launch_count(const vvcb_ctx*) { return 0; }
int vvcb_cu_eval_phases(const vvcb_ctx* ctx, uint64_t ns[8], uint64_t* calls) { if (!ctx || !ns) return VVCB_ERR_ARG; for (int i = 0; i < 8; i++) ns[i] = 0; if (calls) *calls = 0; return VVCB_OK; }
const char* vvcb_last_error(const vvcb_ctx* ctx) { return ctx ? ctx->err : g_createErr; }

int vvcb_create(vvcb_ctx** out, int device, int bit_depth, int ctu_size)
{
  if (!out || bit_depth < 8 || bit_depth > 10 || ctu_size < 32 || ctu_size > 128 || (ctu_size & (ctu_size - 1))) { snprintf(g_createErr, sizeof(g_createErr), "vvcb_create: bad argument"); return VVCB_ERR_ARG; }
  vvcb_ctx* ctx = new vvcb_ctx();
  ctx->bd = bit_depth; ctx->ctu = ctu_size; ctx->depQuant = 1; ctx->width = ctx->height = 0; ctx->remote = nullptr; ctx->err[0] = 0;
  ctx->origP = &ctx->origOwn; ctx->recoP = &ctx->recoOwn;
  if (const char* path = getenv("VVCB_BROKER")) {
    ctx->remote = vvcbc_connect(path, bit_depth, ctu_size, g_createErr, sizeof(g_createErr));
    if (!ctx->remote) { delete ctx; return VVCB_ERR_STATE; }
  }
  *out = ctx;
  return VVCB_OK;
}

void vvcb_destroy(vvcb_ctx* ctx) { if (ctx) { if (ctx->remote) vvcbc_disconnect(ctx->remote); delete ctx; } }

int vvcb_set_option(vvcb_ctx* ctx, int option, int value)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (option == VVCB_OPT_DEP_QUANT && (value == 0 || value == 1)) {
    ctx->depQuant = value;
    if (ctx->remote) return vvcbc_set_option(ctx->remote, option, value, ctx->err, sizeof(ctx->err));
    return VVCB_OK;
  }
  if (option == VVCB_OPT_YIELD_SYNC && (value == 0 || value == 1)) return VVCB_OK;
  FAIL(VVCB_ERR_ARG, "vvcb_set_option: unknown option");
}

int vvcb_frame_alloc(vvcb_ctx* ctx, int width, int height)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_frame_alloc: not available through the broker");
  if (width <= 0 || height <= 0 || (width & 3) || (height & 3)) FAIL(VVCB_ERR_ARG, "vvcb_frame_alloc: bad argument");
  ctx->width = width; ctx->height = height;
  ctx->origP = &ctx->origOwn; ctx->recoP = &ctx->recoOwn;
  (*ctx->origP).assign((size_t)width * height, 0); (*ctx->recoP).assign((size_t)width * height, 0);
  return VVCB_OK;
}

int vvcb_frame_share(vvcb_ctx* dst, vvcb_ctx* src)
{
  if (!dst || !src || src->origOwn.empty()) return VVCB_ERR_STATE;
  dst->origP = &src->origOwn; dst->recoP = &src->recoOwn; dst->width = src->width; dst->height = src->height;
  return VVCB_OK;
}

int vvcb_frame_begin(vvcb_ctx* ctx, const int16_t* orig, int stride, int width, int height)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (!orig || width <= 0 || height <= 0 || stride < width || (width & 3) || (height & 3)) FAIL(VVCB_ERR_ARG, "vvcb_frame_begin: bad argument");
  if (ctx->remote) return vvcbc_frame_begin(ctx->remote, orig, stride, width, height, ctx->err, sizeof(ctx->err));
  int rc = vvcb_frame_alloc(ctx, width, height);
  if (rc) return rc;
  for (int y = 0; y < height; y++) memcpy(&(*ctx->origP)[(size_t)y * width], orig + (size_t)y * stride, width * sizeof(int16_t));
  return VVCB_OK;
}

static int put_rect(vvcb_ctx* ctx, std::vector<int16_t>& plane, const int16_t* src, int stride, int x, int y, int w, int h, const char* who)
{
  if (plane.empty()) FAIL(VVCB_ERR_STATE, "%s: no frame", who);
  if (!src || x < 0 || y < 0 || w <= 0 || h <= 0 || x + w > ctx->width || y + h > ctx->height || stride < w) FAIL(VVCB_ERR_ARG, "%s: rectangle outside the picture", who);
  for (int r = 0; r < h; r++) memcpy(&plane[(size_t)(y + r) * ctx->width + x], src + (size_t)r * stride, w * sizeof(int16_t));
  return VVCB_OK;
}

int vvcb_reco_update(vvcb_ctx* ctx, const int16_t* reco, int stride, int x, int y, int w, int h)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) {
    if (!reco || w <= 0 || h <= 0 || stride < w) FAIL(VVCB_ERR_ARG, "vvcb_reco_update: bad argument");
    std::vector<int16_t> dense((size_t)w * h);
    for (int r = 0; r < h; r++) memcpy(&dense[(size_t)r * w], reco + (size_t)r * stride, w * sizeof(int16_t));
    vvcb_rect rc = { (int16_t)x, (int16_t)y, (int16_t)w, (int16_t)h, 0 };
    return vvcb_reco_update_rects(ctx, &rc, 1, dense.data(), dense.size());
  }
  return put_rect(ctx, (*ctx->recoP), reco, stride, x, y, w, h, "vvcb_reco_update");
}

int vvcb_orig_update(vvcb_ctx* ctx, const int16_t* orig, int stride, int x, int y, int w, int h)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_orig_update: not available through the broker");
  return put_rect(ctx, (*ctx->origP), orig, stride, x, y, w, h, "vvcb_orig_update");
}

int vvcb_reco_update_rects(vvcb_ctx* ctx, const vvcb_rect* rects, int n, const int16_t* samples, size_t n_samples)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && (!rects || !samples))) FAIL(VVCB_ERR_ARG, "vvcb_reco_update_rects: bad argument");
  if (ctx->remote) {
    vvcb_cu_request rq;
    memset(&rq, 0, sizeof(rq));
    rq.rects = rects; rq.n_rects = n; rq.rect_samples = samples; rq.n_rect_samples = n_samples;
    return vvcbc_cu_eval(ctx->remote, &rq, 1, ctx->err, sizeof(ctx->err));
  }
  for (int i = 0; i < n; i++) {
    if (rects[i].w <= 0 || rects[i].h <= 0 || (size_t)rects[i].offset + (size_t)rects[i].w * rects[i].h > n_samples) FAIL(VVCB_ERR_ARG, "vvcb_reco_update_rects: rectangle %d is malformed", i);
    int rc = put_rect(ctx, (*ctx->recoP), samples + rects[i].offset, rects[i].w, rects[i].x, rects[i].y, rects[i].w, rects[i].h, "vvcb_reco_update_rects");
    if (rc) return rc;
  }
  return VVCB_OK;
}

static bool visit_ok(const vvcb_ctx* ctx, const vvcb_rmd_visit& v)
{
  const int w = 1 << v.log2w, h = 1 << v.log2h;
  bool ok = v.log2w >= 2 && v.log2w <= 6 && v.log2h >= 2 && v.log2h <= 6 && v.x >= 0 && v.y >= 0 && (v.x & 3) == 0 && (v.y & 3) == 0 &&
            v.x + w <= ctx->width && v.y + h <= ctx->height && v.n_above <= w / 4 && v.n_above_right <= w / 4 && v.n_left <= h / 4 &&
            v.n_below_left <= h / 4 && v.avail_al <= 1 && v.num_mpm_cand <= 6 &&
            (!(v.avail_al || v.n_above || v.n_above_right) || v.y >= 4) && (!(v.avail_al || v.n_left || v.n_below_left) || v.x >= 4) &&
            v.x + w + 4 * v.n_above_right <= ctx->width && v.y + h + 4 * v.n_below_left <= ctx->height;
  for (int k = 0; k < 6; k++) ok = ok && v.mpm[k] < VVCB_NUM_LUMA_MODE;
  return ok;
}

int vvcb_rmd_eval(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n, vvcb_rmd_result* results, vvcb_rmd_detail* details)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && (!visits || !results))) FAIL(VVCB_ERR_ARG, "vvcb_rmd_eval: bad argument");
  if (ctx->remote) {
    std::vector<vvcb_cu_request> rq(n);
    memset(rq.data(), 0, n * sizeof(vvcb_cu_request));
    for (int i = 0; i < n; i++) { rq[i].visit = &visits[i]; rq[i].want_rmd = 1; rq[i].result = &results[i]; rq[i].detail = details ? &details[i] : nullptr; }
    return vvcbc_cu_eval(ctx->remote, rq.data(), n, ctx->err, sizeof(ctx->err));
  }
  if ((*ctx->origP).empty()) FAIL(VVCB_ERR_STATE, "vvcb_rmd_eval: vvcb_frame_begin has not been called");
  for (int i = 0; i < n; i++) if (!visit_ok(ctx, visits[i])) FAIL(VVCB_ERR_ARG, "vvcb_rmd_eval: visit %d is malformed", i);
  for (int i = 0; i < n; i++)
    orc_rmd_visit((*ctx->origP).data(), ctx->width, (*ctx->recoP).data(), ctx->width, ctx->bd, ctx->ctu, &visits[i], &results[i], details ? &details[i] : nullptr, nullptr);
  return VVCB_OK;
}

int vvcb_rmd_pred_all(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int16_t* pred)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_rmd_pred_all: not available through the broker");
  if (!visit || !pred || !visit_ok(ctx, *visit)) FAIL(VVCB_ERR_ARG, "vvcb_rmd_pred: bad argument");
  vvcb_rmd_result r;
  const int w = 1 << visit->log2w, h = 1 << visit->log2h;
  std::vector<int16_t> all((size_t)VVCB_NUM_SLOTS * w * h, (int16_t)0x7fff);
  std::vector<int16_t> keep(pred, pred + all.size());
  vvcb_rmd_detail det;
  orc_rmd_visit((*ctx->origP).data(), ctx->width, (*ctx->recoP).data(), ctx->width, ctx->bd, ctx->ctu, visit, &r, &det, all.data());
  for (int s = 0; s < VVCB_NUM_SLOTS; s++)
    if (det.sad[s] != VVCB_SAT_NONE) memcpy(pred + (size_t)s * w * h, &all[(size_t)s * w * h], (size_t)w * h * sizeof(int16_t));
  return VVCB_OK;
}

int vvcb_rmd_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visit, int slot, int16_t* pred)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (!visit || !pred || slot < 0 || slot >= VVCB_NUM_SLOTS) FAIL(VVCB_ERR_ARG, "vvcb_rmd_pred: bad argument");
  const int w = 1 << visit->log2w, h = 1 << visit->log2h;
  std::vector<int16_t> all((size_t)VVCB_NUM_SLOTS * w * h);
  int rc = vvcb_rmd_pred_all(ctx, visit, all.data());
  if (rc) return rc;
  memcpy(pred, &all[(size_t)slot * w * h], (size_t)w * h * sizeof(int16_t));
  return VVCB_OK;
}

void vvcb_mts_preselect(const int32_t* sums, int n, int width, int height, int max_cand, uint8_t* selected)
{
  if (n <= 0) return;
  std::vector<int> s(sums, sums + n);
  orc_mts_preselect(s.data(), n, width, height, max_cand, selected);
}

// one TU job on given prediction / residual (dense w*h)
static void tu_chain(vvcb_ctx* ctx, const vvcb_tu_job& j, const int16_t* resi, const int16_t* pred, const vvcb_dq_rates* rates, const vvcb_ctx_states* states,
                     int32_t* coeffOut, int32_t* levelOut, int16_t* recoOut, vvcb_tu_result& r)
{
  const int w = 1 << j.log2w, h = 1 << j.log2h, n = w * h, bd = ctx->bd;
  const bool ts = j.mts_idx == 1;
  std::vector<int32_t> coeff(n), level(n, 0), deq(n, 0);
  std::vector<int16_t> res(n), reco(n);
  if (ts) orc_transform_skip(resi, w, w, h, bd, coeff.data());
  else {
    orc_fwd_transform_ex(resi, w, w, h, bd, j.mts_idx, j.lfnst_idx, coeff.data());
    if (j.lfnst_idx) orc_fwd_lfnst(coeff.data(), w, h, j.intra_mode, j.lfnst_idx);
  }
  memset(&r, 0, sizeof(r));
  r.abs_sum_coeff = orc_abs_sum_for_preselection(coeff.data(), w, h, j.mts_idx);
  if (coeffOut) memcpy(coeffOut, coeff.data(), n * sizeof(int32_t));
  if (!(j.flags & VVCB_TU_QUANT)) return;
  const int qp = j.qp_per * 6 + j.qp_rem;
  if (j.flags & VVCB_TU_DEPQUANT) {
    r.abs_sum_level = orc_dep_quant(coeff.data(), w, h, bd, j.mts_idx, j.lfnst_idx, qp, j.lambda, &rates[j.rate_idx], j.cbf_delta_bits, level.data());
    orc_dep_dequant(level.data(), w, h, bd, qp, deq.data());
  } else if (j.flags & VVCB_TU_RDOQ_TS) {
    r.abs_sum_level = orc_rdoq_ts(coeff.data(), w, h, bd, qp, j.lambda, &rates[j.rate_idx], level.data());
    orc_dequant(level.data(), w, h, bd, j.qp_per, j.qp_rem, 1, deq.data());
  } else {
    r.abs_sum_level = orc_quant_scalar(coeff.data(), w, h, bd, j.qp_per, j.qp_rem, ts, level.data());
    orc_dequant(level.data(), w, h, bd, j.qp_per, j.qp_rem, ts, deq.data());
  }
  if (!ts && j.lfnst_idx) orc_inv_lfnst(deq.data(), w, h, j.intra_mode, j.lfnst_idx);
  if (ts) orc_inv_transform_skip(deq.data(), w, h, bd, res.data(), w);
  else    orc_inv_transform(deq.data(), w, h, bd, j.mts_idx, res.data(), w);
  r.sse = orc_reconstruct_sse(&(*ctx->origP)[(size_t)j.y * ctx->width + j.x], ctx->width, pred, res.data(), w, h, bd, reco.data());
  if ((j.flags & VVCB_TU_RATE) && r.abs_sum_level)
    r.frac_bits = orc_residual_bits(level.data(), w, h, j.mts_idx, (j.flags & VVCB_TU_TS_ALLOWED) != 0, (j.flags & VVCB_TU_MTS_ALLOWED) != 0, ctx->depQuant, &states[j.rate_idx]);
  if (levelOut) memcpy(levelOut, level.data(), n * sizeof(int32_t));
  if (recoOut) memcpy(recoOut, reco.data(), n * sizeof(int16_t));
}

static bool job_ok(const vvcb_ctx* ctx, const vvcb_tu_job& j, size_t n_samples, const void* rates, const void* states, int n_rates)
{
  const size_t sz = (size_t)1 << (j.log2w + j.log2h);
  const bool q = (j.flags & VVCB_TU_QUANT) != 0, dq = q && (j.flags & VVCB_TU_DEPQUANT);
  bool ok = j.log2w >= 2 && j.log2w <= 6 && j.log2h >= 2 && j.log2h <= 6 && j.mts_idx <= 5 && (size_t)j.offset + sz <= n_samples && j.qp_rem >= 0 && j.qp_rem < 6 && j.qp_per >= 0 && j.qp_per < 16;
  if (j.mts_idx >= 1) ok = ok && j.log2w <= 5 && j.log2h <= 5;
  if (q) ok = ok && !(*ctx->origP).empty() && j.x >= 0 && j.y >= 0 && j.x + (1 << j.log2w) <= ctx->width && j.y + (1 << j.log2h) <= ctx->height;
  if (dq) ok = ok && j.mts_idx != 1 && rates && j.rate_idx < n_rates && j.lfnst_idx <= 2 && j.lambda > 0.0;
  if (j.flags & VVCB_TU_RDOQ_TS) ok = ok && q && !dq && j.mts_idx == 1 && rates && j.rate_idx < n_rates && j.lambda > 0.0;
  ok = ok && j.lfnst_idx <= 2 && (j.lfnst_idx == 0 || j.intra_mode < VVCB_NUM_LUMA_MODE);
  if (j.flags & VVCB_TU_RATE) ok = ok && q && states && j.rate_idx < n_rates;
  return ok;
}

int vvcb_tu_eval(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int16_t* resi, const int16_t* pred, size_t n_samples,
                 const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates, int32_t* coeff, int32_t* level, int16_t* reco, vvcb_tu_result* results)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_tu_eval: not available through the broker (use vvcb_tu_eval_pred / vvcb_cu_eval)");
  if (n < 0 || (n > 0 && (!jobs || !results || !resi))) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval: bad argument");
  for (int i = 0; i < n; i++) {
    if (!job_ok(ctx, jobs[i], n_samples, rates, states, n_rates)) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval: job %d is malformed", i);
    if ((jobs[i].flags & VVCB_TU_QUANT) && !pred) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval: VVCB_TU_QUANT needs the prediction samples");
  }
  for (int i = 0; i < n; i++) {
    const size_t o = jobs[i].offset;
    tu_chain(ctx, jobs[i], resi + o, pred ? pred + o : nullptr, rates, states, coeff ? coeff + o : nullptr, level ? level + o : nullptr, reco ? reco + o : nullptr, results[i]);
  }
  return VVCB_OK;
}

static int tu_eval_pred_local(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_tu_src* src, const vvcb_tu_job* jobs, int n,
                              size_t n_samples, const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                              int32_t* coeff, int32_t* level, int16_t* reco, int16_t* pred_out, vvcb_tu_result* results)
{
  if (n < 0 || (n > 0 && (!jobs || !results || !src || !visits || n_visits <= 0))) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval_pred: bad argument");
  if (n == 0) return VVCB_OK;
  if ((*ctx->origP).empty()) FAIL(VVCB_ERR_STATE, "vvcb_tu_eval_pred: vvcb_frame_begin has not been called");
  for (int i = 0; i < n_visits; i++) if (!visit_ok(ctx, visits[i])) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval_pred: visit %d is malformed", i);
  std::map<uint32_t, std::vector<int16_t>> preds;
  std::map<uint32_t, vvcb_rmd_detail> dets;
  for (int i = 0; i < n; i++) {
    if (src[i].visit >= (uint32_t)n_visits || src[i].slot >= VVCB_NUM_SLOTS) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval_pred: source %d is malformed", i);
    const vvcb_rmd_visit& v = visits[src[i].visit];
    if (!job_ok(ctx, jobs[i], n_samples, rates, states, n_rates) || jobs[i].x != v.x || jobs[i].y != v.y || jobs[i].log2w != v.log2w || jobs[i].log2h != v.log2h)
      FAIL(VVCB_ERR_ARG, "vvcb_tu_eval_pred: job %d is malformed", i);
    if (!preds.count(src[i].visit)) {
      const int w = 1 << v.log2w, h = 1 << v.log2h;
      std::vector<int16_t>& p = preds[src[i].visit];
      p.resize((size_t)VVCB_NUM_SLOTS * w * h);
      vvcb_rmd_result r;
      orc_rmd_visit((*ctx->origP).data(), ctx->width, (*ctx->recoP).data(), ctx->width, ctx->bd, ctx->ctu, &v, &r, &dets[src[i].visit], p.data());
    }
    if (dets[src[i].visit].sad[src[i].slot] == VVCB_SAT_NONE) FAIL(VVCB_ERR_ARG, "vvcb_tu_eval_pred: source %d: slot not evaluated for the visit", i);
  }
  for (int i = 0; i < n; i++) {
    const vvcb_tu_job& j = jobs[i];
    const int w = 1 << j.log2w, h = 1 << j.log2h;
    const int16_t* p = &preds[src[i].visit][(size_t)src[i].slot * w * h];
    std::vector<int16_t> resi((size_t)w * h);
    for (int y = 0; y < h; y++) for (int x = 0; x < w; x++) resi[y * w + x] = (int16_t)((*ctx->origP)[(size_t)(j.y + y) * ctx->width + j.x + x] - p[y * w + x]);
    const size_t o = j.offset;
    tu_chain(ctx, j, resi.data(), p, rates, states, coeff ? coeff + o : nullptr, level ? level + o : nullptr, reco ? reco + o : nullptr, results[i]);
    if (pred_out) memcpy(pred_out + o, p, (size_t)w * h * sizeof(int16_t));
  }
  return VVCB_OK;
}

int vvcb_tu_eval_pred(vvcb_ctx* ctx, const vvcb_rmd_visit* visits, int n_visits, const vvcb_tu_src* src, const vvcb_tu_job* jobs, int n,
                      size_t n_samples, const vvcb_dq_rates* rates, const vvcb_ctx_states* states, int n_rates,
                      int32_t* coeff, int32_t* level, int16_t* reco, int16_t* pred_out, vvcb_tu_result* results)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_tu_eval_pred: not available through the broker (use vvcb_cu_eval)");
  return tu_eval_pred_local(ctx, visits, n_visits, src, jobs, n, n_samples, rates, states, n_rates, coeff, level, reco, pred_out, results);
}

int vvcb_residual_bits(vvcb_ctx* ctx, const vvcb_tu_job* jobs, int n, const int32_t* levels, size_t n_samples, const vvcb_ctx_states* states, int n_states, uint64_t* bits)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote) FAIL(VVCB_ERR_STATE, "vvcb_residual_bits: not available through the broker");
  if (n < 0 || (n > 0 && (!jobs || !levels || !states || !bits || n_states <= 0))) FAIL(VVCB_ERR_ARG, "vvcb_residual_bits: bad argument");
  for (int i = 0; i < n; i++) {
    const vvcb_tu_job& j = jobs[i];
    const int w = 1 << j.log2w, h = 1 << j.log2h;
    if (j.rate_idx >= n_states || (size_t)j.offset + (size_t)w * h > n_samples) FAIL(VVCB_ERR_ARG, "vvcb_residual_bits: job %d is malformed", i);
    bool any = false;
    for (int k = 0; k < w * h; k++) any = any || levels[j.offset + k] != 0;
    bits[i] = any ? orc_residual_bits(levels + j.offset, w, h, j.mts_idx, (j.flags & VVCB_TU_TS_ALLOWED) != 0, (j.flags & VVCB_TU_MTS_ALLOWED) != 0, ctx->depQuant, &states[j.rate_idx]) : 0;
  }
  return VVCB_OK;
}

// profiling entry points the shims reference: nothing to time here
int vvcb_kernel_timing(vvcb_ctx* ctx, int) { return ctx ? VVCB_OK : VVCB_ERR_ARG; }
int vvcb_kernel_times(vvcb_ctx* ctx, float ms[3], int* launches) { if (!ctx || !ms) return VVCB_ERR_ARG; ms[0] = ms[1] = ms[2] = 0.f; if (launches) *launches = 0; return VVCB_OK; }
int vvcb_tu_kernel_times(vvcb_ctx* ctx, float ms[4], int* calls) { if (!ctx || !ms) return VVCB_ERR_ARG; ms[0] = ms[1] = ms[2] = ms[3] = 0.f; if (calls) *calls = 0; return VVCB_OK; }

int vvcb_reco_from_orig(vvcb_ctx* ctx)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (ctx->remote || (*ctx->origP).empty()) FAIL(VVCB_ERR_STATE, "vvcb_reco_from_orig: no frame owned by the context");
  *ctx->recoP = *ctx->origP;
  return VVCB_OK;
}

int vvcb_cu_eval(vvcb_ctx* ctx, vvcb_cu_request* reqs, int n)
{
  if (!ctx) return VVCB_ERR_ARG;
  if (n < 0 || (n > 0 && !reqs)) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: bad argument");
  if (ctx->remote) return vvcbc_cu_eval(ctx->remote, reqs, n, ctx->err, sizeof(ctx->err));
  std::lock_guard<std::mutex> lock(g_oracleMutex);
  for (int i = 0; i < n; i++) {                      // reconstruction first: requests of one call belong to different pictures
    vvcb_cu_request& q = reqs[i];
    if (q.n_rects) { int rc = vvcb_reco_update_rects(ctx, q.rects, q.n_rects, q.rect_samples, q.n_rect_samples); if (rc) return rc; }
  }
  for (int i = 0; i < n; i++) {
    vvcb_cu_request& q = reqs[i];
    if ((q.want_rmd || q.n_jobs || q.n_autos) && !q.visit) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: request %d has no visit", i);
    if (q.want_rmd) {
      if (!q.result) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: request %d wants the lists but gives no result pointer", i);
      int rc = vvcb_rmd_eval(ctx, q.visit, 1, q.result, q.detail);
      if (rc) return rc;
    }
    if (q.n_jobs) {
      if (!q.jobs || !q.slots || !q.tu_results) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: request %d: jobs without slots / results", i);
      std::vector<vvcb_tu_src> src(q.n_jobs);
      for (int k = 0; k < q.n_jobs; k++) { src[k].visit = 0; src[k].slot = q.slots[k]; }
      const size_t ns = (size_t)q.n_jobs << (q.visit->log2w + q.visit->log2h);
      int rc = tu_eval_pred_local(ctx, q.visit, 1, src.data(), q.jobs, q.n_jobs, ns, q.rates, q.states, 1, nullptr, q.level, q.reco, q.pred, q.tu_results);
      if (rc) return rc;
    }
    if (q.n_autos) {
      if (!q.want_rmd || !q.autos || q.max_auto <= 0 || !q.n_auto || !q.auto_slot || !q.auto_tmpl || !q.auto_results) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: request %d is malformed (templates)", i);
      for (int k = 0; k < q.n_autos; k++) if ((q.autos[k].modes & VVCB_AUTO_REGULAR) && !q.detail) FAIL(VVCB_ERR_ARG, "vvcb_cu_eval: request %d is malformed (templates)", i);
      std::vector<vvcb_tu_job> jobs(q.max_auto);
      const int cnt = vvcb_expand_autos(*q.visit, *q.result, q.detail, q.autos, q.n_autos, q.max_auto, jobs.data(), q.auto_slot, q.auto_tmpl);
      *q.n_auto = cnt;
      if (cnt) {
        std::vector<vvcb_tu_src> src(cnt);
        for (int k = 0; k < cnt; k++) { src[k].visit = 0; src[k].slot = q.auto_slot[k]; }
        const size_t ns = (size_t)cnt << (q.visit->log2w + q.visit->log2h);
        int rc = tu_eval_pred_local(ctx, q.visit, 1, src.data(), jobs.data(), cnt, ns, q.rates, q.states, 1, nullptr, q.auto_level, q.auto_reco, q.auto_pred, q.auto_results);
        if (rc) return rc;
      }
    }
  }
  return VVCB_OK;
}

} // extern "C"
