// mc_chroma_emul.cpp - CPU replay of me_mc_chroma_kernel, the 4:2:0 chroma motion-compensation + SSE kernel of cucd_me_mc_chroma
// (TEST HARNESS, not a product path).
//
// me_mc_chroma_kernel (csrc/me_kernels.cu) is a thin shell around the __host__ __device__ code of csrc/me_core.cuh: the host plan
// (me_mcc_job, me_mcc_plan) and the phases me_mcc_stage / _hor / _ver / _sse.  This file replays every CTA the way the kernel runs it,
// each phase for all 256 thread ids between the barriers, on poisoned shared memory, so that `pytest -m "not gpu"` can compare its
// arithmetic and its packing with the checker (tests/test_emulation_mc_chroma.py).
#include <algorithm>
#include <cstdint>
#include <vector>
#include "../../include/cucudecide.h"
#include "me_core.cuh"

using namespace cucd;

// The host plan of cucd_me_mc_chroma and, per CTA, the phases of me_mc_chroma_kernel for all 256 thread ids.  cur[plane]: the current
// Cb / Cr plane (curStride); refPlane[2 s + plane]: the first sample of slot s's padded Cb / Cr plane (refStride[s], marginX[s],
// marginY[s]).  sse[2 i + plane]; pred: Cb then Cr block per candidate.  Returns the CTA count, -1 if a CTA overflows a cap.
extern "C" int emul_mc_chroma(int bitDepth, const int16_t* const* cur, int curStride, const int16_t* const* refPlane, const int32_t* refStride,
                              const int* marginX, const int* marginY, int n, const cucd_mc_desc* desc, uint32_t* sse, int16_t* pred) {
  std::vector<McJob> jobs(n), sorted(n);
  long long predOff = 0;
  for (int i = 0; i < n; i++) {
    const cucd_mc_desc& d = desc[i];
    const int cx = d.x >> 1, cy = d.y >> 1, cw = d.w >> 1, ch = d.h >> 1;
    int nl = 0, slot[2], mvx[2], mvy[2], stride[2], mX[2], mY[2];
    for (int l = 0; l < 2; l++) {
      if (d.ref_idx[l] < 0) continue;
      const int s = d.ref_idx[l];
      slot[nl] = s; mvx[nl] = d.mvx[l]; mvy[nl] = d.mvy[l]; stride[nl] = refStride[s]; mX[nl] = marginX[s]; mY[nl] = marginY[s]; nl++;
    }
    jobs[i] = me_mcc_job(cy * curStride + cx, cx, cy, cw, ch, nl, slot, mvx, mvy, stride, mX, mY, i, predOff);
    predOff += 2LL * cw * ch;
  }
  std::vector<int32_t> ctaFirst(n + 1);
  const int nCta = me_mcc_plan(n, jobs.data(), sorted.data(), ctaFirst.data());
  std::vector<int16_t> sCur(kMcCurCap), sWin(kMcWinCap), sTmp(kMcTmpCap);
  int sSum[2 * kMcMaxCand];
  for (int b = 0; b < nCta; b++) {
    std::fill(sCur.begin(), sCur.end(), (int16_t)0x5a5a); std::fill(sWin.begin(), sWin.end(), (int16_t)0x5a5a); std::fill(sTmp.begin(), sTmp.end(), (int16_t)0x5a5a);
    std::fill(sSum, sSum + 2 * kMcMaxCand, 0x5a5a5a5a);
    const McJob* J = sorted.data() + ctaFirst[b];
    const McGeo g = me_mcc_geo(J[0].w, J[0].h, J[0].nl, ctaFirst[b + 1] - ctaFirst[b], bitDepth);
    if (g.n > kMcMaxCand || 2 * g.n * g.wh > kMcCurCap || 2 * g.n * g.nl * g.win > kMcWinCap || 2 * g.n * g.nl * g.tmp > kMcTmpCap) return -1;
    for (int tid = 0; tid < 256; tid++) { if (tid < 2 * g.n) sSum[tid] = 0; me_mcc_stage(tid, g, J, cur, curStride, refPlane, refStride, sCur.data(), sWin.data()); }
    for (int tid = 0; tid < 256; tid++) me_mcc_hor(tid, g, J, sWin.data(), sTmp.data());
    for (int tid = 0; tid < 256; tid++) me_mcc_ver(tid, g, J, sTmp.data(), sWin.data(), pred);
    for (int tid = 0; tid < 256; tid++) me_mcc_sse(tid, g, sCur.data(), sWin.data(), sSum);
    for (int tid = 0; tid < 2 * g.n; tid++) sse[2 * J[tid >> 1].outIndex + (tid & 1)] = (uint32_t)sSum[tid];
  }
  return nCta;
}
