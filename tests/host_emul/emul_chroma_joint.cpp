// TEST INFRASTRUCTURE -- the kernels of vvcb_chroma_joint_tu_eval (vvc_intra_b200/csrc/vvcb_chroma.cuh, vvcb_tu.cuh, vvcb_dq.cuh,
// vvcb_rate.cuh) on host threads through cuda_emul.h, for tests/test_chroma_joint_tu_eval.py: the kernel source itself, checked against
// the C chain without a GPU.  Includes emul_chroma.cpp (the harness of emul_rmd.cpp and the chroma kernels) and adds one entry point;
// built by the test into a temporary directory.
#include "emul_chroma.cpp"

// vvcb_chroma_joint_tu_eval's kernels on host threads, in the order chroma_joint_tu_chunk (vvcb_api.cu) launches them:
// chroma_tu_pred_kernel<true>, the TU chain with the residual-output pass (pass 0, the chroma dependent quantiser on prices derived from
// the starting models, pass 1, the chroma rate kernel on the carried models) and chroma_joint_kernel.  Outputs as
// vvcb_chroma_joint_tu_eval returns them (2 w*h per candidate at jobs[i].offset); depQuant: the slice flag the rate kernel follows.
extern "C" int emul_chroma_joint_tu_eval(const int16_t* const planes[4], int cstride, const int16_t* luma, int lstride, int bd, int ctu,
                                         int depQuant, const vvcb_chroma_visit* visits, int nVisits, const vvcb_chroma_joint_tu_job* jobs, int n,
                                         const vvcb_chroma_joint_ctx_states* states, size_t nSamples, int32_t* level, int16_t* reco,
                                         int16_t* pred, vvcb_chroma_joint_tu_result* results)
{
  static Rom rom;
  static TrRom trRom;
  static DqRom dqRom;
  static RateRom rr;
  fill_rom(rom); fill_tr_rom(trRom); fill_dq_rom(dqRom);
  for (int i = 0; i < 512; i++) rr.binFracBits[i] = kBinFracBits[i];
  std::vector<vvcb_tu_job> tj(n);
  std::vector<vvcb_chroma_ctx_states> cst(n);
  std::vector<vvcb_bin_model> jm((size_t)3 * n);
  for (int i = 0; i < n; i++) {
    const vvcb_chroma_joint_tu_job& j = jobs[i];
    const vvcb_chroma_visit& v = visits[j.visit];
    if (j.flags & (VVCB_TU_DEPQUANT | VVCB_TU_RATE)) {
      cst[i] = states[j.rate_idx].chroma;
      for (int k = 0; k < 3; k++) jm[(size_t)3 * i + k] = states[j.rate_idx].joint[k];
    } else {
      memset(&cst[i], 0, sizeof(cst[i]));
      memset(&jm[(size_t)3 * i], 0, 3 * sizeof(vvcb_bin_model));
    }
    vvcb_tu_job& t = tj[i];
    memset(&t, 0, sizeof(t));
    t.x = v.x; t.y = v.y; t.log2w = v.log2w; t.log2h = v.log2h; t.flags = j.flags; t.qp_per = j.qp_per; t.qp_rem = j.qp_rem;
    t.offset = j.offset; t.rate_idx = (uint16_t)i; t.lambda = j.lambda;
  }
  std::vector<int16_t> resi(nSamples);
  std::vector<int32_t> dqCoeff(nSamples), dqDeq(nSamples, 0);
  std::vector<vvcb_tu_result> res(n);
  std::vector<vvcb_dq_rates> rates(n);
  std::vector<DqRateTab> tabs(n);
  std::vector<uint64_t> sse((size_t)2 * n, 0);
  std::vector<uint8_t> cbf(n, 0);
  std::vector<uint32_t> bits((size_t)3 * n, 0);
  memset(level, 0, nSamples * sizeof(int32_t));
  ChromaTuPredParams Q = {};
  Q.planes.visits = visits; Q.planes.n = nVisits;
  for (int c = 0; c < 2; c++) { Q.planes.orig[c] = planes[c]; Q.planes.reco[c] = planes[2 + c]; }
  Q.planes.cstride = cstride; Q.planes.luma = luma; Q.planes.lstride = lstride; Q.planes.bd = bd; Q.planes.ctu = ctu; Q.planes.rom = &rom;
  Q.joint = jobs; Q.n = n; Q.cbJobs = tj.data(); Q.states = cst.data(); Q.pred = pred; Q.resi = resi.data(); Q.frac = rr.binFracBits;
  emu_launch(2, kChromaWarps * 32, [&] { chroma_tu_pred_kernel<true>(Q); });
  std::vector<int> smallList, largeList, order, rateOrder;
  for (int i = 0; i < n; i++) {
    (tj[i].log2w + tj[i].log2h <= 8 ? smallList : largeList).push_back(i);
    if (tj[i].flags & VVCB_TU_DEPQUANT) order.push_back(i);
    if (tj[i].flags & VVCB_TU_RATE) rateOrder.push_back(i);
  }
  TuParams P;
  P.jobs = tj.data(); P.list = nullptr; P.n = 0; P.resi = resi.data(); P.pred = pred; P.coeff = nullptr; P.level = level; P.reco = reco;
  P.results = res.data(); P.orig = planes[0]; P.stride = cstride; P.bd = bd; P.rom = &trRom;
  P.dqCoeff = dqCoeff.data(); P.dqDeq = dqDeq.data(); P.phase = 0;
  auto launch_tu = [&](TuParams T) {
    if (!smallList.empty()) { T.list = smallList.data(); T.n = (int)smallList.size(); emu_launch(2, kTuThreads, [&] { tu_eval_kernel<32, true>(T); }); }
    if (!largeList.empty()) { T.list = largeList.data(); T.n = (int)largeList.size(); emu_launch(2, kTuThreads, [&] { tu_eval_kernel<128, true>(T); }); }
  };
  launch_tu(P);
  const int nDq = (int)order.size();
  if (nDq) {
    emu_launch((n * kChromaResidualModels + 127) / 128, 128, [&] { chroma_rates_from_states_kernel(cst.data(), n, &rr, rates.data()); });
    emu_launch(n, 32, [&] { dq_rate_kernel(rates.data(), n, tabs.data()); });
    const int grid = 2;
    std::vector<uint8_t> scratch((size_t)grid * kDqGroups * kDqSlotBytes);
    std::vector<int> firstRaw(nDq), orderSorted(nDq), firstSorted(nDq), binCount(kDqBins, 0);
    emu_launch(2, kDqThreads, [&] { dq_first_kernel(tj.data(), order.data(), nDq, dqCoeff.data(), &dqRom, bd, firstRaw.data()); });
    const bool sortJobs = nDq > 48;            // both orders run at the scale of the test sets (the product sorts above 2048 jobs)
    if (sortJobs) {
      const int sortGrid = (nDq + kDqSortPerBlock - 1) / kDqSortPerBlock;
      emu_launch(sortGrid, kDqSortThreads, [&] { dq_hist_kernel(firstRaw.data(), nDq, binCount.data()); });
      emu_launch(1, 32, [&] { dq_scan_kernel(binCount.data()); });
      emu_launch(sortGrid, kDqSortThreads, [&] { dq_scatter_kernel(order.data(), firstRaw.data(), nDq, binCount.data(), orderSorted.data(), firstSorted.data()); });
    }
    DqParams D;
    D.jobs = tj.data(); D.order = sortJobs ? orderSorted.data() : order.data(); D.firstPos = sortJobs ? firstSorted.data() : firstRaw.data(); D.n = nDq;
    D.coeff = dqCoeff.data(); D.level = level; D.deq = dqDeq.data(); D.results = res.data();
    D.rates = rates.data(); D.tabs = tabs.data(); D.rom = &dqRom; D.scratch = scratch.data(); D.bd = bd; D.sparse = !sortJobs;
    emu_launch(grid, kDqThreads, [&] { dq_kernel<true>(D); });
    P.phase = 1;
    launch_tu(P);
  }
  if (!rateOrder.empty()) {
    RateParams R;
    R.jobs = tj.data(); R.order = rateOrder.data(); R.n = (int)rateOrder.size(); R.level = level; R.results = res.data();
    R.states = reinterpret_cast<const vvcb_ctx_states*>(cst.data()); R.statesOut = reinterpret_cast<vvcb_ctx_states*>(cst.data());
    R.rom = &dqRom; R.rate = &rr; R.depQuant = depQuant;
    emu_launch(2, kRateThreads, [&] { rate_kernel<true>(R); });
  }
  ChromaJointParams F;
  F.jobs = jobs; F.n = n; F.visits = visits; F.tuJobs = tj.data(); F.res = res.data(); F.pred = pred; F.reco = reco;
  F.orig[0] = planes[0]; F.orig[1] = planes[1]; F.cstride = cstride; F.bd = bd;
  F.states = cst.data(); F.joint = jm.data(); F.sse = sse.data(); F.cbf = cbf.data(); F.bits = bits.data(); F.frac = rr.binFracBits;
  emu_launch(2, 128, [&] { chroma_joint_kernel(F); });
  for (int i = 0; i < n; i++) {
    vvcb_chroma_joint_tu_result& r = results[i];
    memset(&r, 0, sizeof(r));
    const bool rate = (jobs[i].flags & VVCB_TU_RATE) != 0;
    r.res = res[i];
    if (!rate) r.res.frac_bits = 0;
    r.sse[0] = sse[2 * i]; r.sse[1] = sse[2 * i + 1];
    r.cbf = cbf[i];
    if (rate) { r.cbf_bits[0] = bits[3 * i]; r.cbf_bits[1] = bits[3 * i + 1]; r.joint_bits = bits[3 * i + 2]; }
  }
  return 0;
}
