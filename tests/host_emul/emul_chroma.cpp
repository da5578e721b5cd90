// TEST INFRASTRUCTURE -- chroma_eval_kernel (vvc_intra_b200/csrc/vvcb_chroma.cuh) on host threads through cuda_emul.h, for
// tests/test_chroma_eval.py: the kernel source itself, checked against the oracle without a GPU.  Includes the harness of emul_rmd.cpp
// (thread-local CUDA built-ins, emu_launch) and adds one entry point; built by the test into a temporary directory.
#include "emul_rmd.cpp"
#include "../../vvc_intra_b200/csrc/vvcb_chroma.cuh"

// planes: Cb orig, Cr orig, Cb reco, Cr reco (stride cstride); luma: the luma reconstruction (stride lstride).  pred_out (optional):
// per visit 8 x 2 blocks of w*h, one visit after another, as vvcb_chroma_eval returns them.
extern "C" int emul_chroma_eval(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                                const vvcb_chroma_visit* visits, int n, int16_t* pred_out, vvcb_chroma_result* results)
{
  static Rom rom;
  fill_rom(rom);
  std::vector<uint32_t> off((size_t)n);
  size_t total = 0;
  for (int i = 0; i < n; i++) { off[i] = (uint32_t)total; total += (size_t)VVCB_CHROMA_CANDS * 2 << (visits[i].log2w + visits[i].log2h); }
  if (pred_out) memset(pred_out, 0, total * sizeof(int16_t));
  ChromaParams P;
  P.visits = visits; P.n = n; P.results = results; P.predOut = pred_out; P.predOff = off.data();
  for (int c = 0; c < 2; c++) { P.orig[c] = planes[c]; P.reco[c] = planes[2 + c]; }
  P.cstride = cstride; P.luma = luma; P.lstride = lstride; P.bd = bd; P.ctu = ctu; P.rom = &rom;
  emu_launch(2, kChromaWarps * 32, [&] { chroma_eval_kernel(P); });
  return 0;
}
