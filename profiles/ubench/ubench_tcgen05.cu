// ubench_tcgen05.cu - measurements that size the tensor-core RMD design (not a product path):
//   A. what tcgen05.ld ... .pack::16b returns           B. TMEM read throughput (LDTM) per SM
//   C. kind::i8 with UNSIGNED A and B is exact          D. tcgen05.mma issue rate, M128 N64 K32
// build: nvcc -gencode arch=compute_100a,code=sm_100a -O3 -I../../fast-cu-decision-hevc_b200/csrc ubench_tcgen05.cu -o ubench_tcgen05
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <cuda_runtime.h>
#include "satd_tc.cuh"
using namespace cucd::tc;

#define LD32_ASM(PACK) \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32" PACK ".b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n" \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]), \
        "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), \
        "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), \
        "=r"(v[30]), "=r"(v[31]) : "r"(addr) : "memory")
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t* v) { LD32_ASM(""); }
__device__ __forceinline__ void tmem_ld32_pack(uint32_t addr, uint32_t* v) { LD32_ASM(".pack::16b"); }

// ---- A: pack semantics ---------------------------------------------------------------------------
__global__ void k_pack(uint32_t* out) {
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0) tmem_alloc(&slot, 64);
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t base = slot + ((uint32_t)(warp * 32) << 16);
  uint32_t v[16];
  for (int h = 0; h < 2; h++) {
    for (int c = 0; c < 16; c++) v[c] = (uint32_t)(0x100 * (h * 16 + c) + lane) | ((uint32_t)(0xA000 + h * 16 + c) << 16);
    tmem_st16(base + h * 16, v);
    tmem_st_wait();
  }
  tc_fence_before(); __syncthreads(); tc_fence_after();
  tmem_ld16_pack(base, v); tmem_ld_wait();
  for (int c = 0; c < 16; c++) out[threadIdx.x * 16 + c] = v[c];
  tc_fence_before(); __syncthreads();
  if (warp == 0) tmem_dealloc(slot, 64);
}

// ---- B: LDTM throughput ----------------------------------------------------------------------------
template <int MODE>
__global__ void k_ldtm(long long* cycles, uint32_t* sink, int iters) {
  __shared__ uint32_t slot;
  const int warp = threadIdx.x >> 5;
  if (warp == 0) tmem_alloc(&slot, 512);
  tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t base = slot + ((uint32_t)((warp & 3) * 32) << 16);
  uint32_t acc = 0;
  __syncthreads();
  const long long t0 = clock64();
  for (int i = 0; i < iters; i++) {
    uint32_t v[32];
    const uint32_t addr = base + ((i * 64) & 255) + (warp >> 2) * 32 % 64;
    if (MODE == 0) tmem_ld32(addr, v); else if (MODE == 1) tmem_ld32_pack(addr, v); else { tmem_ld16(addr, v); tmem_ld16(addr + 16, v + 16); }
    tmem_ld_wait();
#pragma unroll
    for (int k = 0; k < 32; k += 8) acc += v[k];
  }
  __syncthreads();
  const long long t1 = clock64();
  if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
  sink[blockIdx.x * blockDim.x + threadIdx.x] = acc;
  tc_fence_before(); __syncthreads();
  if (warp == 0) tmem_dealloc(slot, 512);
}

// ---- C/D: u8 x u8 MMA, correctness + rate -----------------------------------------------------------
__device__ __forceinline__ uint32_t idesc_u8u8(int M, int N) {
  uint32_t d = 0; d |= 2u << 4; d |= (uint32_t)(N >> 3) << 17; d |= (uint32_t)(M >> 4) << 24; return d;   // a_format = b_format = 0 (unsigned 8 bit)
}
__global__ void k_mma(const uint8_t* A /*128x32 row-major*/, const uint8_t* B /*64x32 row-major*/, uint32_t* D /*128x64*/, long long* cycles, int reps) {
  extern __shared__ __align__(128) unsigned char sm[];
  unsigned char* sA = sm; unsigned char* sB = sm + 4096;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + 4096 + 2048); uint32_t* slot = reinterpret_cast<uint32_t*>(mbar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) { mbar_init(mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
  if (warp == 0) tmem_alloc(slot, 64);
  for (int i = tid; i < 128 * 32; i += blockDim.x) { const int r = i >> 5, k = i & 31; sA[(k >> 4) * 2048 + (r >> 3) * 128 + (r & 7) * 16 + (k & 15)] = A[i]; }
  for (int i = tid; i < 64 * 32; i += blockDim.x) { const int r = i >> 5, k = i & 31; sB[(k >> 4) * 1024 + (r >> 3) * 128 + (r & 7) * 16 + (k & 15)] = B[i]; }
  fence_async_smem(); tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t tmem = *slot;
  const uint64_t dA = make_desc(smem_u32(sA), 2048, 128), dB = make_desc(smem_u32(sB), 1024, 128);
  const uint32_t id = idesc_u8u8(128, 64);
  long long t0 = 0, t1 = 0;
  if (tid == 0) {
    t0 = clock64();
    for (int r = 0; r < reps; r++) mma_i8(tmem, dA, dB, id, 0u);
    mma_commit(mbar);
  }
  mbar_wait(mbar, 0); tc_fence_after();
  if (tid == 0) { t1 = clock64(); cycles[0] = t1 - t0; }
  for (int c = 0; c < 4; c++) {
    uint32_t v[16];
    tmem_ld16(tmem + ((uint32_t)((warp & 3) * 32) << 16) + c * 16, v); tmem_ld_wait();
    for (int k = 0; k < 16; k++) D[tid * 64 + c * 16 + k] = v[k];
  }
  tc_fence_before(); __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 64);
}


// ---- E: A operand in TMEM (one row per lane, K bytes packed 4 per 32-bit column) ---------------------
__global__ void k_mma_ts(const uint8_t* A /*128x64 row-major*/, const uint8_t* B /*64x64 row-major*/, uint32_t* D /*128x64*/) {
  extern __shared__ __align__(128) unsigned char sm[];
  unsigned char* sB = sm;
  uint64_t* mbar = reinterpret_cast<uint64_t*>(sm + 4096); uint32_t* slot = reinterpret_cast<uint32_t*>(mbar + 1);
  const int tid = threadIdx.x, warp = tid >> 5;
  if (tid == 0) { mbar_init(mbar, 1); asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
  if (warp == 0) tmem_alloc(slot, 128);
  for (int i = tid; i < 64 * 64; i += blockDim.x) { const int r = i >> 6, k = i & 63; sB[(k >> 4) * 1024 + (r >> 3) * 128 + (r & 7) * 16 + (k & 15)] = B[i]; }
  fence_async_smem(); tc_fence_before(); __syncthreads(); tc_fence_after();
  const uint32_t tmem = *slot;
  const uint32_t lane0 = (uint32_t)((warp & 3) * 32) << 16;
  uint32_t v[16];
  for (int c = 0; c < 16; c++) v[c] = reinterpret_cast<const uint32_t*>(A + tid * 64)[c];
  tmem_st16(tmem + lane0 + 64, v);                 // A at columns 64..79, D at 0..63
  tmem_st_wait();
  tc_fence_before(); __syncthreads(); tc_fence_after();
  if (tid == 0) {
    const uint64_t dB = make_desc(smem_u32(sB), 1024, 128);
    const uint32_t id = idesc_u8u8(128, 64);
    mma_i8_ts(tmem, tmem + 64, dB, id, 0u);
    mma_i8_ts(tmem, tmem + 64 + 8, dB + ((2 * 1024) >> 4), id, 1u);
    mma_commit(mbar);
  }
  mbar_wait(mbar, 0); tc_fence_after();
  for (int c = 0; c < 4; c++) {
    tmem_ld16(tmem + lane0 + c * 16, v); tmem_ld_wait();
    for (int k = 0; k < 16; k++) D[tid * 64 + c * 16 + k] = v[k];
  }
  tc_fence_before(); __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, 128);
}

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)
int main() {
  uint32_t* dOut; CK(cudaMalloc(&dOut, 128 * 16 * 4));
  k_pack<<<1, 128>>>(dOut); CK(cudaDeviceSynchronize());
  std::vector<uint32_t> h(128 * 16); CK(cudaMemcpy(h.data(), dOut, h.size() * 4, cudaMemcpyDeviceToHost));
  printf("A pack::16b: stored col c = (0x100*c + lane) | (0xA000+c)<<16, 32 columns; ld x16.pack lane 3:\n  ");
  for (int c = 0; c < 16; c++) printf("%08x ", h[3 * 16 + c]); printf("\n");

  long long* dCyc; uint32_t* dSink; CK(cudaMalloc(&dCyc, 8 * 148 * 8)); CK(cudaMalloc(&dSink, 148 * 8 * 1024 * 4));
  const int iters = 2000;
  for (int mode = 0; mode < 3; mode++) for (int warps = 4; warps <= 16; warps *= 2) {
    if (mode == 0) k_ldtm<0><<<148, warps * 32>>>(dCyc, dSink, iters); else if (mode == 1) k_ldtm<1><<<148, warps * 32>>>(dCyc, dSink, iters); else k_ldtm<2><<<148, warps * 32>>>(dCyc, dSink, iters);
    CK(cudaDeviceSynchronize());
    long long c; CK(cudaMemcpy(&c, dCyc, 8, cudaMemcpyDeviceToHost));
    const double colsPerLd = mode == 1 ? 64 : 32;
    printf("B ldtm mode %d (%s) warps %2d: %lld cycles / %d iters = %.1f cyc per warp-load, %.1f TMEM bytes/cycle/SM, %.2f regs/cycle/SM\n", mode,
           mode == 0 ? "x32" : mode == 1 ? "x32.pack16" : "2 x x16", warps, c, iters, (double)c / iters, warps * 32.0 * colsPerLd * 4 * iters / c, warps * 32.0 * 32 * iters / c);
  }

  std::vector<uint8_t> hA(128 * 32), hB(64 * 32);
  srand(7); for (auto& x : hA) x = rand() & 255; for (auto& x : hB) x = rand() & 255;
  uint8_t *dA, *dB; uint32_t* dD; CK(cudaMalloc(&dA, hA.size())); CK(cudaMalloc(&dB, hB.size())); CK(cudaMalloc(&dD, 128 * 64 * 4));
  CK(cudaMemcpy(dA, hA.data(), hA.size(), cudaMemcpyHostToDevice)); CK(cudaMemcpy(dB, hB.data(), hB.size(), cudaMemcpyHostToDevice));
  for (int reps : {1, 64, 1024}) {
    k_mma<<<1, 128, 8192>>>(dA, dB, dD, dCyc, reps); CK(cudaDeviceSynchronize());
    long long c; CK(cudaMemcpy(&c, dCyc, 8, cudaMemcpyDeviceToHost));
    std::vector<uint32_t> hD(128 * 64); CK(cudaMemcpy(hD.data(), dD, hD.size() * 4, cudaMemcpyDeviceToHost));
    int bad = 0;
    for (int r = 0; r < 128; r++) for (int j = 0; j < 64; j++) { uint32_t s = 0; for (int k = 0; k < 32; k++) s += (uint32_t)hA[r * 32 + k] * hB[j * 32 + k]; if (s != hD[r * 64 + j]) bad++; }
    printf("C/D u8xu8 M128 N64 K32 x %d: %lld cycles (%.1f per MMA), mismatches %d\n", reps, c, (double)c / reps, bad);
  }
  {
    std::vector<uint8_t> hA2(128 * 64), hB2(64 * 64);
    for (auto& x : hA2) x = rand() & 255; for (auto& x : hB2) x = rand() & 255;
    uint8_t *dA2, *dB2; CK(cudaMalloc(&dA2, hA2.size())); CK(cudaMalloc(&dB2, hB2.size()));
    CK(cudaMemcpy(dA2, hA2.data(), hA2.size(), cudaMemcpyHostToDevice)); CK(cudaMemcpy(dB2, hB2.data(), hB2.size(), cudaMemcpyHostToDevice));
    k_mma_ts<<<1, 128, 8192>>>(dA2, dB2, dD); CK(cudaDeviceSynchronize());
    std::vector<uint32_t> hD(128 * 64); CK(cudaMemcpy(hD.data(), dD, hD.size() * 4, cudaMemcpyDeviceToHost));
    int bad = 0;
    for (int r = 0; r < 128; r++) for (int j = 0; j < 64; j++) { uint32_t s = 0; for (int k = 0; k < 64; k++) s += (uint32_t)hA2[r * 64 + k] * hB2[j * 64 + k]; if (s != hD[r * 64 + j]) bad++; }
    printf("E A-in-TMEM u8xu8 M128 N64 K64: mismatches %d (row0: got %u %u want-first %u)\n", bad, hD[0], hD[1], 0u);
  }
  return 0;
}
