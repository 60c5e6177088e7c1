// tc2_skew.cu - how far apart the four warps of a row group run inside one mode round of rmd_frame_tc2_kernel (development aid).
// build: profiles/ubench/build.sh tc2_skew tc2_skew.cu -DCUCD_TC2_WARPSKEW
// Events of round am = 4 of the first pass, lane 0 of warps 0..3 of row group 0, clock64 of the SM:
//   0 before wait MMA1 | 1 after it | 2 after epilogue 1 + tcgen05.st | 3 before arrive(A) | 4 after arrive(A) (+ MMA 2 issue in warp 0)
//   5 after window / weight staging | 6 after wait MMA2 | 7 after arrive(B) (+ MMA 1 issue in warp 0) | 8 after epilogue 2
//   9 / 10: events 0 / 1 of the NEXT round (am = 3)
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include "../../fast-cu-decision-hevc_b200/csrc/rmd_tc2_kernels.cu"
using namespace cucd;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
int main() {
  const int W = 1920, H = 1080, P = 16, pitch = 1920, ctusPerRow = 30, ctusPerPic = 510, total = P * ctusPerPic;
  std::vector<int16_t> h((size_t)P * pitch * H);
  srand(1); for (auto& v : h) v = rand() & 255;
  int16_t *dOrg, *dRec; uint32_t* dOut; int8_t* dHad; uint8_t* dTab; long long* dDbg;
  CK(cudaMalloc(&dOrg, h.size() * 2)); CK(cudaMalloc(&dRec, h.size() * 2)); CK(cudaMalloc(&dOut, (size_t)total * 341 * 35 * 4));
  CK(cudaMalloc(&dHad, 16384)); uint8_t* dPrep; CK(cudaMalloc(&dPrep, rmd_tc2_prep_bytes(total))); CK(cudaMalloc(&dTab, tc2::kWinTableBytes + tc2::kN4TableBytes));
  CK(cudaMemcpy(dOrg, h.data(), h.size() * 2, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dRec, h.data(), h.size() * 2, cudaMemcpyHostToDevice));
  std::vector<uint8_t> tab(tc2::kWinTableBytes + tc2::kN4TableBytes);
  tc2::fill_win_tables(tab.data()); tc2::fill_n4_tables(tab.data() + tc2::kWinTableBytes);
  CK(cudaMemcpy(dTab, tab.data(), tab.size(), cudaMemcpyHostToDevice));
  {
    std::vector<int8_t> had(16384, 0);     // layout of hadamard_operands_kernel (rmd_kernels.cu)
    for (int j = 0; j < 64; j++)
      for (int k = 0; k < 64; k++) {
        const int y = k >> 3, x = k & 7, off = tc2::umma_off64(j, k);
        const int s8 = (__builtin_popcount((j >> 3) & y) + __builtin_popcount((j & 7) & x)) & 1;
        had[off] = (int8_t)(s8 ? -1 : 1); had[4096 + off] = (int8_t)(s8 ? 1 : -1);
        const int q = j >> 4, u = (j >> 2) & 3, v = j & 3, qk = (y >> 2) * 2 + (x >> 2);
        const int s4 = (__builtin_popcount(u & (y & 3)) + __builtin_popcount(v & (x & 3))) & 1;
        const int e = q == qk ? (s4 ? -1 : 1) : 0;
        had[8192 + off] = (int8_t)e; had[12288 + off] = (int8_t)(-e);
      }
    CK(cudaMemcpy(dHad, had.data(), had.size(), cudaMemcpyHostToDevice));
  }
  const int u2 = (total + 1) / 2, u4 = (total + 3) / 4, blocks = 2 * u4 + 3 * u2;
  CK(cudaMalloc(&dDbg, (size_t)blocks * 64 * 8)); CK(cudaMemset(dDbg, 0, (size_t)blocks * 64 * 8));
  CK(cudaMemcpyToSymbol(g_tc2Skew, &dDbg, sizeof(dDbg)));
  FrameSource fs; fs.org = dOrg; fs.rec = dRec; fs.orgPicStride = (long long)pitch * H; fs.recPicStride = fs.orgPicStride; fs.orgStride = pitch; fs.recStride = pitch;
  fs.W = W; fs.H = H; fs.ctusPerRow = ctusPerRow; fs.ctusPerPic = ctusPerPic; fs.out = dOut; fs.outPacked = nullptr; fs.needed = nullptr;
  CK(configure_rmd_tc2_kernels());
  for (int it = 0; it < 2; it++) CK(launch_rmd_frames_tc2(fs, P, 1, dTab, dTab + tc2::kWinTableBytes, dHad, dPrep, 0, nullptr));
  CK(cudaDeviceSynchronize());
  std::vector<long long> d((size_t)blocks * 64); CK(cudaMemcpy(d.data(), dDbg, d.size() * 8, cudaMemcpyDeviceToHost));
  // N = 8 blocks: indices [2*u4 + u2, 2*u4 + 2*u2)
  const char* names[11] = {"pre-wait1", "wait1 done", "E1+st", "pre-arrA", "arrA(+iss2)", "staged", "wait2 done", "arrB(+iss1)", "E2 done", "next pre-wait1", "next wait1 done"};
  for (int kind = 0; kind < 2; kind++) {
    const int b0 = kind == 0 ? 2 * u4 + u2 : 2 * u4, b1 = b0 + u2;
    double avg[4][11] = {{0}}; double spreadA = 0, spreadB = 0, mma2lat = 0, mma1lat = 0; int n = 0;
    for (int b = b0 + 300; b < b1 - 300; b++) {
      const long long* t = &d[(size_t)b * 64];
      if (!t[0]) continue;
      n++;
      long long t0 = t[0];
      for (int w = 0; w < 4; w++) for (int e = 0; e < 11; e++) avg[w][e] += (double)(t[w * 16 + e] - t0);
      long long lastA = 0, firstA = 1LL << 62, lastB = 0, firstB = 1LL << 62, done2 = 1LL << 62, done1n = 0;
      for (int w = 0; w < 4; w++) {
        lastA = std::max(lastA, t[w * 16 + 3]); firstA = std::min(firstA, t[w * 16 + 3]);
        lastB = std::max(lastB, t[w * 16 + 6]); firstB = std::min(firstB, t[w * 16 + 6]);
        done2 = std::min(done2, t[w * 16 + 6]);
      }
      spreadA += (double)(lastA - firstA); spreadB += (double)(lastB - firstB);
      mma2lat += (double)(done2 - lastA);
    }
    printf("%s CTAs (%d sampled), round am = 4, cycles relative to warp 0's first stamp:\n", kind == 0 ? "N = 8" : "N = 16", n);
    for (int w = 0; w < 4; w++) { printf("  warp %d:", w); for (int e = 0; e < 11; e++) printf(" %s %6.0f |", names[e], avg[w][e] / n); printf("\n"); }
    printf("  spread of the four warps at arrive(A): %.0f cycles; earliest 'wait MMA2 done' minus LAST arrive(A): %.0f cycles (= tcgen05.wait::st + fence + issue + MMA 2 + commit)\n",
           spreadA / n, mma2lat / n);
  }
  return 0;
}
