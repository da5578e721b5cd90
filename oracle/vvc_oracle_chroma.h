/*
 * TEST INFRASTRUCTURE -- the chroma part of the oracle (vvc_oracle_chroma.c): candidates of the chroma intra search, their
 * prediction and SAD / SATD.  Parity status: UNPINNED (restated from H.266 and the cited reference lines).
 */
#ifndef VVC_ORACLE_CHROMA_H
#define VVC_ORACLE_CHROMA_H
#include "vvc_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

void orc_chroma_ref_fill(const int16_t* reco, int stride, int x, int y, int w, int h, int bd,
                         int avail_al, int n_above, int n_above_right, int n_left, int n_below_left, int16_t* top, int16_t* left);
void orc_chroma_ipa_init(int w, int h, int mode, orc_ipa* p);
void orc_chroma_pred_angular(const int16_t* top, const int16_t* left, int w, int h, int bd, const orc_ipa* p, int16_t* pred);
void orc_cclm_luma(const int16_t* luma, int lstride, int w, int h, int avail_l, int ctu_top, int n_top, int n_left,
                   int16_t* ds, int16_t* ds_top, int16_t* ds_left);
void orc_cclm_params(int lm, int w, int h, int bd, int avail_t, int avail_l, int n_ar, int n_bl,
                     const int16_t* ds_top, const int16_t* ds_left, const int16_t* c_top, const int16_t* c_left, int* a, int* k, int* b);
void orc_cclm_pred(const int16_t* ds, int w, int h, int bd, int a, int k, int b, int16_t* pred);
void orc_chroma_cand_modes(int dm_mode, uint8_t modes[VVCB_CHROMA_CANDS]);
void orc_chroma_visit(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                      const vvcb_chroma_visit* v, vvcb_chroma_result* out, int16_t* pred_out);
void orc_chroma_batch(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                      const vvcb_chroma_visit* v, int n, vvcb_chroma_result* out, int16_t* pred_out);

#ifdef __cplusplus
}
#endif
#endif
