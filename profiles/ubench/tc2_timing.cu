// tc2_timing.cu - clock64 timeline of rmd_frame_tc2_kernel CTAs (development aid, not a product path).
// build: nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -DCUCD_TC2_TIMING -I../../fast-cu-decision-hevc_b200/csrc tc2_timing.cu -o tc2_timing
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <algorithm>
#include "../../fast-cu-decision-hevc_b200/csrc/rmd_tc2_kernels.cu"

using namespace cucd;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
int main(int argc, char** argv) {
  const int W = 1920, H = 1080, P = argc > 1 ? atoi(argv[1]) : 4, pitch = 1920;
  const int ctusPerRow = 30, ctusPerPic = 30 * 17, total = P * ctusPerPic;
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
  CK(cudaMemcpyToSymbol(g_tc2Dbg, &dDbg, sizeof(dDbg)));
  FrameSource fs; fs.org = dOrg; fs.rec = dRec; fs.orgPicStride = (long long)pitch * H; fs.recPicStride = fs.orgPicStride; fs.orgStride = pitch; fs.recStride = pitch;
  fs.W = W; fs.H = H; fs.ctusPerRow = ctusPerRow; fs.ctusPerPic = ctusPerPic; fs.out = dOut; fs.outPacked = nullptr; fs.needed = nullptr;
  CK(configure_rmd_tc2_kernels());
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int it = 0; it < 3; it++) {
    cudaEventRecord(e0);
    CK(launch_rmd_frames_tc2(fs, P, 1, dTab, dTab + tc2::kWinTableBytes, dHad, dPrep, 0, nullptr));
    cudaEventRecord(e1); CK(cudaDeviceSynchronize());
    float ms; cudaEventElapsedTime(&ms, e0, e1); printf("launch %d: %.3f ms (%d CTUs, %.2f M CTU/s)\n", it, ms, total, total / ms / 1e3);
  }
  std::vector<long long> d((size_t)blocks * 64); CK(cudaMemcpy(d.data(), dDbg, d.size() * 8, cudaMemcpyDeviceToHost));
  for (int l = 6; l >= 2; l--) {
    double pro = 0, pass = 0, tail = 0, setup = 0, rounds[17] = {0}; int n = 0;
    for (int b = 0; b < blocks; b++) {
      const long long* t = &d[(size_t)b * 64];
      if (t[4] != l) continue;
      n++; pro += t[1] - t[0]; pass += t[2] - t[1]; tail += t[3] - t[2]; setup += t[8] - t[1];
      for (int r = 0; r < 17; r++) rounds[r] += t[9 + r] - t[8 + r];
    }
    if (!n) continue;
    printf("N=%2d: %5d CTAs  prologue %7.0f  passes %8.0f (first-pass setup %6.0f)  copy-out %6.0f  clk;  rounds am=8..-8:", 1 << l, n, pro / n, pass / n, setup / n, tail / n);
    for (int r = 0; r < 17; r++) printf(" %4.0f", rounds[r] / n);
    printf("\n");
    {
      double g[8] = {0};
      for (int b = 0; b < blocks; b++) {
        const long long* t = &d[(size_t)b * 64];
        if (t[4] != l) continue;
        g[0] += t[50] - t[0]; g[1] += t[54] - t[50]; g[2] += t[55] - t[54]; g[3] += t[1] - t[55];
        g[6] += t[56] - t[1]; g[7] += t[57] - t[56];
      }
      { double h[4] = {0}; for (int b = 0; b < blocks; b++) { const long long* t = &d[(size_t)b * 64]; if (t[4] != l) continue; h[0] += t[58] - t[0]; h[1] += t[59] - t[58]; h[2] += t[60] - t[59]; h[3] += t[50] - t[60]; }
        printf("      first phase: tmem alloc %5.0f | issue loads %5.0f | zero + first load lands %5.0f | second table store + sync %5.0f\n", h[0] / n, h[1] / n, h[2] / n, h[3] / n); }
      printf("      prologue: alloc+tables+zero+sync %5.0f | PU states %5.0f | fences+CTA barrier %5.0f | wait for the border copies %5.0f || pass set-up: source tile %5.0f | operands+planar/DC %5.0f\n",
             g[0] / n, g[1] / n, g[2] / n, g[3] / n, g[6] / n, g[7] / n);
    }
    for (int base = 30; base <= 40; base += 10) {
      double seg[8] = {0};
      for (int b = 0; b < blocks; b++) { const long long* t = &d[(size_t)b * 64]; if (t[4] != l) continue; for (int k = 0; k < 8; k++) seg[k] += t[base + k + 1] - t[base + k]; }
      printf("      round am=%2d: wait MMA1 %4.0f | epilogue 1 + st %4.0f | projected refs %4.0f | st wait + barrier + issue MMA2 %4.0f | stage %4.0f | wait MMA2 %4.0f | barrier + issue MMA1 %4.0f | epilogue 2 %4.0f\n",
             base == 30 ? 4 : -4, seg[0] / n, seg[1] / n, seg[2] / n, seg[3] / n, seg[4] / n, seg[5] / n, seg[6] / n, seg[7] / n);
    }
  }
  return 0;
}
