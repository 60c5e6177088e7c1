// mc_emul.cpp - CPU replay of me_mc_kernel, the motion-compensation + distortion kernel of cucd_me_mc_cost (TEST HARNESS, not a
// product path).
//
// me_mc_kernel (csrc/me_kernels.cu) is a thin shell around the __host__ __device__ code of csrc/me_core.cuh: the host plan (me_mc_job,
// me_mc_plan: candidates sorted by class and cut into CTAs), the phases me_mc_stage / me_mc_hor / me_mc_ver and subpel_small_dist.
// This file replays every CTA the way the kernel runs it, each phase for all 256 thread ids between the barriers, on poisoned shared
// memory, so that `pytest -m "not gpu"` can compare its arithmetic and its packing with the checker (tests/test_emulation_mc.py).
#include <algorithm>
#include <cstdint>
#include <vector>
#include "../../include/cucudecide.h"
#include "me_core.cuh"

using namespace cucd;

// ---- motion compensation + distortion of inter candidates: the host plan of cucd_me_mc_cost and, per CTA, the phases of me_mc_kernel
// for all 256 thread ids.  refPlane[s]: the first sample of padded plane s (marginX[s], marginY[s], refStride[s]); returns the CTA count.
extern "C" int emul_mc_cost(int bitDepth, const int16_t* cur, int curStride, const int16_t* const* refPlane, const int32_t* refStride, const int* marginX,
                            const int* marginY, int n, const cucd_mc_desc* desc, uint32_t* dist, int16_t* pred) {
  std::vector<McJob> jobs(n), sorted(n);
  long long predOff = 0;
  for (int i = 0; i < n; i++) {
    const cucd_mc_desc& d = desc[i];
    int nl = 0, slot[2], mvx[2], mvy[2], stride[2], mX[2], mY[2];
    for (int l = 0; l < 2; l++) {
      if (d.ref_idx[l] < 0) continue;
      const int s = d.ref_idx[l];
      slot[nl] = s; mvx[nl] = d.mvx[l]; mvy[nl] = d.mvy[l]; stride[nl] = refStride[s]; mX[nl] = marginX[s]; mY[nl] = marginY[s]; nl++;
    }
    jobs[i] = me_mc_job(d.y * curStride + d.x, d.x, d.y, d.w, d.h, nl, slot, mvx, mvy, stride, mX, mY, d.use_hadamard, i, predOff);
    predOff += (long long)d.w * d.h;
  }
  std::vector<int32_t> ctaFirst(n + 1);
  const int nCta = me_mc_plan(n, jobs.data(), sorted.data(), ctaFirst.data());
  std::vector<int16_t> sCur(kMcCurCap), sWin(kMcWinCap), sTmp(kMcTmpCap);
  int sSum[kMcMaxCand];
  for (int b = 0; b < nCta; b++) {
    std::fill(sCur.begin(), sCur.end(), (int16_t)0x5a5a); std::fill(sWin.begin(), sWin.end(), (int16_t)0x5a5a); std::fill(sTmp.begin(), sTmp.end(), (int16_t)0x5a5a);
    const McJob* J = sorted.data() + ctaFirst[b];
    const McGeo g = me_mc_geo(J[0].w, J[0].h, J[0].nl, ctaFirst[b + 1] - ctaFirst[b], bitDepth);
    if (g.n > kMcMaxCand || g.n * g.wh > kMcCurCap || g.n * g.nl * g.win > kMcWinCap || g.n * g.nl * g.tmp > kMcTmpCap) return -1;
    for (int tid = 0; tid < 256; tid++) { if (tid < g.n) sSum[tid] = 0; me_mc_stage(tid, g, J, cur, curStride, refPlane, refStride, sCur.data(), sWin.data()); }
    for (int tid = 0; tid < 256; tid++) me_mc_hor(tid, g, J, sWin.data(), sTmp.data());
    for (int tid = 0; tid < 256; tid++) me_mc_ver(tid, g, J, sTmp.data(), sWin.data(), pred);
    for (int tid = 0; tid < 256; tid++) subpel_small_dist(tid, subpel_geo(g.w, g.h, g.bd), g.n, J[0].had, sCur.data(), sWin.data(), sSum, g.wh);
    for (int tid = 0; tid < g.n; tid++) dist[J[tid].outIndex] = (uint32_t)sSum[tid] >> (bitDepth - 8);
  }
  return nCta;
}
