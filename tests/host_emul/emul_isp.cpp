// TEST INFRASTRUCTURE -- isp_pred_kernel (vvc_intra_b200/csrc/vvcb_rmd.cuh) on host threads through cuda_emul.h, for
// tests/test_isp_eval.py: the kernel source itself, checked against the oracle chain without a GPU.  Includes the harness of
// emul_rmd.cpp (thread-local CUDA built-ins, emu_launch) and adds one entry point; built by the test into a temporary directory.
#include "emul_rmd.cpp"

// Step k of n candidates.  cand: n rows of (x, y, cu_w, cu_h, hor, mode, avail_al, n_above, n_above_right, n_left, n_below_left, offset);
// cu_reco: the candidates' reconstructions (blocks in coding order at offset, each dense w*h), read for the lines of block k > 0;
// pred / resi: block k of every candidate that has one is written at offset + k*w*h.
extern "C" int emul_isp_pred(const int16_t* orig, const int16_t* reco, int stride, int bd, const int32_t* cand, int n, int k,
                             const int16_t* cu_reco, int16_t* pred, int16_t* resi)
{
  static Rom rom;
  fill_rom(rom);
  std::vector<IspCand> cands(n);
  std::vector<int> list;
  for (int i = 0; i < n; i++) {
    const int32_t* c = cand + 12 * i;
    IspCand& d = cands[i];
    const int cuW = c[2], cuH = c[3], hor = c[4];
    const int split = hor ? cuH : cuW, other = hor ? cuW : cuH;       // PartitionerImpl::getTUIntraSubPartitions
    const int size = vmax(split >> 2, other < 16 ? 16 / other : 1);
    d.x = (int16_t)c[0]; d.y = (int16_t)c[1]; d.cuW = (int16_t)cuW; d.cuH = (int16_t)cuH;
    d.bw = (int16_t)(hor ? cuW : size); d.bh = (int16_t)(hor ? size : cuH);
    d.topLen = (int16_t)(cuW + d.bw); d.leftLen = (int16_t)(cuH + d.bh);
    d.hor = (uint8_t)hor; d.nParts = (uint8_t)(split / size); d.mode = (uint8_t)c[5];
    d.availAl = (uint8_t)c[6]; d.nAbove = (uint8_t)c[7]; d.nAboveRight = (uint8_t)c[8]; d.nLeft = (uint8_t)c[9]; d.nBelowLeft = (uint8_t)c[10];
    d.offset = (uint32_t)c[11];
    d.p = make_mode_param_isp(cuW, cuH, d.bw, d.bh, d.mode);
    if (d.nParts > k) list.push_back(i);
  }
  std::vector<vvcb_tu_job> jobs(n);
  std::vector<vvcb_tu_result> prev(n);
  std::vector<IspState> state(n);
  memset(jobs.data(), 0, sizeof(vvcb_tu_job) * n);
  memset(prev.data(), 0, sizeof(vvcb_tu_result) * n);
  memset(state.data(), 0, sizeof(IspState) * n);
  IspPredParams Q;
  Q.cands = cands.data(); Q.list = list.data(); Q.n = (int)list.size(); Q.k = k;
  Q.jobs = jobs.data(); Q.prev = prev.data(); Q.state = state.data();
  Q.pred = pred; Q.resi = resi; Q.cuReco = cu_reco; Q.orig = orig; Q.reco = reco; Q.stride = stride; Q.bd = bd;
  Q.rom = &rom; Q.frac = kBinFracBits;
  emu_launch(4, kIspPredWarps * 32, [&] { isp_pred_kernel(Q); });
  return 0;
}
