// rmd_variants.cu - times one frame-RMD kernel source on a 16-picture 1080p batch (development aid, not a product path).
// The kernel source is compiled into the binary, so schedule variants are selected with -D switches at build time:
//   nvcc -std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -DKERNEL=2 [-DCUCD_V_...=..] -I../../fast-cu-decision-hevc_b200/csrc rmd_variants.cu -o v_xxx
// KERNEL=2: rmd_frame_tc2_kernel (8-bit content, kind::i8); KERNEL=3: rmd_frame_tc3_kernel (10-bit content, kind::f16).
// Prints the mean launch time and a checksum of the cost tables (variants of one kernel must print the same checksum).
// KERNEL=2 takes a third argument: full (default: border pre-pass + RMD kernel, as the library launches them), rmd (the RMD kernel
// alone, on images the pre-pass wrote once before the timing: what a free pre-pass would give) or prep (the pre-pass alone).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>
#ifndef KERNEL
#define KERNEL 2
#endif
#if KERNEL == 2
#include "../../fast-cu-decision-hevc_b200/csrc/rmd_tc2_kernels.cu"
#else
#include "../../fast-cu-decision-hevc_b200/csrc/rmd_tc3_kernels.cu"
#endif

using namespace cucd;
#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
int main(int argc, char** argv) {
  const int W = 1920, H = 1080, P = argc > 1 ? atoi(argv[1]) : 16, reps = argc > 2 ? atoi(argv[2]) : 10, pitch = 1920;
  const int bd = KERNEL == 2 ? 8 : 10;
  const int ctusPerRow = 30, ctusPerPic = 30 * 17, total = P * ctusPerPic;
  std::vector<int16_t> h((size_t)P * pitch * H), hr(h.size());
  srand(1);
  // blocky texture + noise, like the bench's synthetic content (pure noise would make every mode equally bad)
  for (int p = 0; p < P; p++)
    for (int y = 0; y < H; y++)
      for (int x = 0; x < W; x++) {
        const unsigned hsh = (unsigned)((y / 8) * 7919 + (x / 8) * 104729 + p * 31) * 2654435761u;
        int v = (int)((hsh >> 24) & 255) * 3 / 5 + 40 + (rand() % 13) - 6;
        v = v < 0 ? 0 : (v > 255 ? 255 : v);
        h[((size_t)p * H + y) * pitch + x] = (int16_t)(v << (bd - 8) | (rand() & ((1 << (bd - 8)) - 1)));
        hr[((size_t)p * H + y) * pitch + x] = (int16_t)(((v + (rand() % 5) - 2) & 255) << (bd - 8));
      }
  int16_t *dOrg, *dRec; uint32_t* dOut;
  CK(cudaMalloc(&dOrg, h.size() * 2)); CK(cudaMalloc(&dRec, h.size() * 2)); CK(cudaMalloc(&dOut, (size_t)total * 341 * 35 * 4));
  CK(cudaMemcpy(dOrg, h.data(), h.size() * 2, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dRec, hr.data(), h.size() * 2, cudaMemcpyHostToDevice));
  FrameSource fs; fs.org = dOrg; fs.rec = dRec; fs.orgPicStride = (long long)pitch * H; fs.recPicStride = fs.orgPicStride; fs.orgStride = pitch; fs.recStride = pitch;
  fs.W = W; fs.H = H; fs.ctusPerRow = ctusPerRow; fs.ctusPerPic = ctusPerPic; fs.out = dOut; fs.outPacked = nullptr; fs.needed = nullptr;
#if KERNEL == 2
  int8_t* dHad; uint8_t* dTab;
  CK(cudaMalloc(&dHad, 16384)); CK(cudaMalloc(&dTab, tc2::kWinTableBytes + tc2::kN4TableBytes));
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
  CK(configure_rmd_tc2_kernels());
  uint8_t* dPrep;
  CK(cudaMalloc(&dPrep, rmd_tc2_prep_bytes(total)));
  CK(cudaMemset(dOut, 0, (size_t)total * 341 * 35 * 4));
  const char* mode = argc > 3 ? argv[3] : "full";
  CK(launch_rmd_border_prep(fs, P, 1, dPrep, 0, nullptr));
  auto launch = [&]() {
    if (!strcmp(mode, "prep")) return launch_rmd_border_prep(fs, P, 1, dPrep, 0, nullptr);
    if (!strcmp(mode, "rmd")) return launch_rmd_frame_tc2(fs, P, 1, dTab, dTab + tc2::kWinTableBytes, dHad, dPrep, 0, nullptr);
    return launch_rmd_frames_tc2(fs, P, 1, dTab, dTab + tc2::kWinTableBytes, dHad, dPrep, 0, nullptr);
  };
#else
  uint8_t* dTab;
  std::vector<uint8_t> tab(tc3::kWinTableBytes16 + tc3::kN4TableBytes16 + tc3::kHadBytes16);
  tc3::fill_win_tables16(tab.data()); tc3::fill_n4_tables16(tab.data() + tc3::kWinTableBytes16); tc3::fill_had_tables16(tab.data() + tc3::kWinTableBytes16 + tc3::kN4TableBytes16);
  CK(cudaMalloc(&dTab, tab.size())); CK(cudaMemcpy(dTab, tab.data(), tab.size(), cudaMemcpyHostToDevice));
  CK(configure_rmd_tc3_kernels());
  auto launch = [&]() { return launch_rmd_frames_tc3(fs, P, bd, 1, dTab, dTab + tc3::kWinTableBytes16, dTab + tc3::kWinTableBytes16 + tc3::kN4TableBytes16, 0, nullptr); };
#endif
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int it = 0; it < 3; it++) CK(launch());
  CK(cudaDeviceSynchronize());
  cudaEventRecord(e0);
  for (int it = 0; it < reps; it++) CK(launch());
  cudaEventRecord(e1); CK(cudaDeviceSynchronize());
  float ms; cudaEventElapsedTime(&ms, e0, e1); ms /= reps;
  std::vector<uint32_t> out((size_t)total * 341 * 35);
  CK(cudaMemcpy(out.data(), dOut, out.size() * 4, cudaMemcpyDeviceToHost));
  unsigned long long sum = 0;
  for (size_t i = 0; i < out.size(); i++) sum = sum * 1000003ull + out[i];
  printf("%s%s%s: %.4f ms per %d-picture launch (%d CTUs, %.3f M CTU/s), checksum %016llx\n", argv[0], KERNEL == 2 ? " " : "", KERNEL == 2 ? (argc > 3 ? argv[3] : "full") : "", ms, P, total, total / ms / 1e3, sum);
  return 0;
}
