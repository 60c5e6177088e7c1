// satd_tc_exp.cu - stand-alone check of the tcgen05 (kind::i8) Hadamard SATD building block of
// satd_tc.cuh: 8x8 tiles of 8-bit source and prediction in, (sum|H(o-p)| + 2) >> 2 per tile out.
// A round-1 experiment kept for reference (not part of libcucudecide.so): the product's rmd_frame_tc2_kernel uses the same
// building block.  Stand-alone program: checks the kernel against a CPU Hadamard and prints the kernel time.
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -I../../fast-cu-decision-hevc_b200/csrc satd_tc_exp.cu -o satd_tc_exp
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "satd_tc.cuh"
enum { CUCD_OK = 0, CUCD_ERR_INVALID = -1, CUCD_ERR_CUDA = -3, CUCD_ERR_NOMEM = -4 };

namespace cucd {
using namespace tc;

__global__ void __launch_bounds__(128)
satd_tc_exp_kernel(const uint8_t* __restrict__ org, const uint8_t* __restrict__ pred, int nGroups, uint32_t* __restrict__ out) {
  __shared__ __align__(128) uint8_t sAO[4 * 2048];
  __shared__ __align__(128) uint8_t sAP[4 * 2048];
  __shared__ __align__(128) int8_t sBpos[4096];
  __shared__ __align__(128) int8_t sBneg[4096];
  __shared__ __align__(8) uint64_t mbar;
  __shared__ uint32_t tmemSlot;
  const int tid = threadIdx.x, warp = tid >> 5;

  fill_hadamard64(sBpos, +1, tid, 128);
  fill_hadamard64(sBneg, -1, tid, 128);
  if (tid == 0) { mbar_init(&mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
  if (warp == 0) tmem_alloc(&tmemSlot, 64);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmemBase = tmemSlot;
  const uint32_t idesc = make_idesc_i8(128, 64, 0, 1);
  const uint64_t dAO = make_desc(smem_u32(sAO), 2048, 128), dAP = make_desc(smem_u32(sAP), 2048, 128);
  const uint64_t dBp = make_desc(smem_u32(sBpos), 1024, 128), dBn = make_desc(smem_u32(sBneg), 1024, 128);
  uint32_t parity = 0;

  for (int g = blockIdx.x; g < nGroups; g += gridDim.x) {
    const size_t row = (size_t)g * 128 + tid;
    const uint4* po = reinterpret_cast<const uint4*>(org + row * 64);
    const uint4* pp = reinterpret_cast<const uint4*>(pred + row * 64);
    const int off = (tid >> 3) * 128 + (tid & 7) * 16;
#pragma unroll
    for (int c = 0; c < 4; c++) {
      *reinterpret_cast<uint4*>(sAO + c * 2048 + off) = po[c];
      *reinterpret_cast<uint4*>(sAP + c * 2048 + off) = pp[c];
    }
    fence_async_smem();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after();
      // K = 64 bytes per operand = 2 instructions of K = 32 (2 chunks of 16 bytes each)
      mma_i8(tmemBase, dAO, dBp, idesc, 0u);
      mma_i8(tmemBase, dAO + ((2 * 2048) >> 4), dBp + ((2 * 1024) >> 4), idesc, 1u);
      mma_i8(tmemBase, dAP, dBn, idesc, 1u);
      mma_i8(tmemBase, dAP + ((2 * 2048) >> 4), dBn + ((2 * 1024) >> 4), idesc, 1u);
      mma_commit(&mbar);
    }
    mbar_wait(&mbar, parity);
    parity ^= 1u;
    tc_fence_after();
    uint32_t acc = 0;
#pragma unroll
    for (int q = 0; q < 4; q++) {
      uint32_t v[16];
      tmem_ld16(tmemBase + ((uint32_t)(warp * 32) << 16) + q * 16, v);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 16; i++) acc += (uint32_t)abs((int)v[i]);
    }
    out[row] = (acc + 2u) >> 2;
    tc_fence_before();
    __syncthreads();
  }
  if (warp == 0) tmem_dealloc(tmemBase, 64);
}

}  // namespace cucd

static int exp_satd_tc(const uint8_t* org, const uint8_t* pred, int nTiles, uint32_t* satd, int iters, float* avg_ms) {
  if (!org || !pred || !satd || nTiles <= 0 || (nTiles & 127) || iters < 1) return CUCD_ERR_INVALID;
  uint8_t *dO = nullptr, *dP = nullptr; uint32_t* dS = nullptr;
  const size_t bytes = (size_t)nTiles * 64;
  if (cudaMalloc(&dO, bytes) != cudaSuccess || cudaMalloc(&dP, bytes) != cudaSuccess || cudaMalloc(&dS, (size_t)nTiles * 4) != cudaSuccess) return CUCD_ERR_NOMEM;
  cudaMemcpy(dO, org, bytes, cudaMemcpyHostToDevice);
  cudaMemcpy(dP, pred, bytes, cudaMemcpyHostToDevice);
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  const int groups = nTiles / 128;
  const int grid = groups < 148 * 8 ? groups : 148 * 8;
  cucd::satd_tc_exp_kernel<<<grid, 128>>>(dO, dP, groups, dS);
  cudaEventRecord(e0);
  for (int i = 0; i < iters; i++) cucd::satd_tc_exp_kernel<<<grid, 128>>>(dO, dP, groups, dS);
  cudaEventRecord(e1);
  cudaError_t e = cudaDeviceSynchronize();
  float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
  if (avg_ms) *avg_ms = ms / iters;
  cudaMemcpy(satd, dS, (size_t)nTiles * 4, cudaMemcpyDeviceToHost);
  cudaFree(dO); cudaFree(dP); cudaFree(dS); cudaEventDestroy(e0); cudaEventDestroy(e1);
  return e == cudaSuccess ? CUCD_OK : CUCD_ERR_CUDA;
}

static uint32_t cpu_satd8x8(const uint8_t* o, const uint8_t* p) {      // xCalcHADs8x8 (TComRdCost.cpp:1439-1534) as a plain matrix product
  int d[64], t[64];
  for (int i = 0; i < 64; i++) d[i] = (int)o[i] - (int)p[i];
  for (int u = 0; u < 8; u++) for (int x = 0; x < 8; x++) { int a = 0; for (int y = 0; y < 8; y++) a += (__builtin_popcount(u & y) & 1) ? -d[y * 8 + x] : d[y * 8 + x]; t[u * 8 + x] = a; }
  uint32_t sum = 0;
  for (int u = 0; u < 8; u++) for (int v = 0; v < 8; v++) { int a = 0; for (int x = 0; x < 8; x++) a += (__builtin_popcount(v & x) & 1) ? -t[u * 8 + x] : t[u * 8 + x]; sum += (uint32_t)abs(a); }
  return (sum + 2) >> 2;
}
int main() {
  const int n = 128 * 40;
  std::vector<uint8_t> org((size_t)n * 64), pred((size_t)n * 64);
  srand(5);
  for (auto& v : org) v = (uint8_t)(rand() & 255);
  for (auto& v : pred) v = (uint8_t)(rand() & 255);
  for (int i = 0; i < 128 * 64; i++) { org[i] = 255; pred[i] = 0; }
  std::vector<uint32_t> got(n);
  float ms = 0;
  if (exp_satd_tc(org.data(), pred.data(), n, got.data(), 3, &ms) != CUCD_OK) { printf("kernel failed\n"); return 1; }
  for (int k = 0; k < n; k++) if (got[k] != cpu_satd8x8(&org[(size_t)k * 64], &pred[(size_t)k * 64])) { printf("MISMATCH at tile %d\n", k); return 1; }
  printf("tensor-core SATD: %d tiles bit-exact, %.1f us per launch\n", n, ms * 1e3);
  return 0;
}
