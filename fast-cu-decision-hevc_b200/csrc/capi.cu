// capi.cu - lifecycle and the frame path of the C ABI (include/cucudecide.h): device buffers, pinned staging, streams, the
// two-pass feature pipeline with the host TCM fit in between (persistent worker pool, begin / end split), the pipelined
// host-buffer call cuCUDecide_frames.  The batch entry points live in capi_batch.cu.  There is no CPU compute path: every
// entry point either runs the CUDA kernels or fails.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include "handle.h"
#include "rmd_tc2.cuh"
#include "rmd_tc3.cuh"
#include "tcm_host.h"

using namespace cucd;

static_assert(kPackedCtuBytes == CUCD_PACKED_CTU_BYTES && kPackedU16Off == CUCD_PACKED_U16_OFFSET && kPackedB13Off == CUCD_PACKED_B13_OFFSET,
              "kernel-side packed cost layout must match include/cucudecide.h");

namespace cucd {
std::string g_createError;

// Registers EXACTLY [ptr, ptr + bytes): rounding the range out to pages would make the first / last bytes of neighbouring heap
// blocks part of a registration, and a later transfer of such a neighbour - a partially registered range - fails with
// cudaErrorInvalidValue.  A request that overlaps ranges this handle registered earlier (a reference plane with its margins
// after the bare plane, say) replaces them by the union.
bool pin_host_range(cucd_handle* h, const void* ptr, size_t bytes) {
  if (!ptr || !bytes) return false;
  uintptr_t lo = (uintptr_t)ptr, hi = lo + bytes;
  for (const auto& r : h->pins) if (r.first <= lo && hi <= r.second) return true;
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, ptr) == cudaSuccess && at.type == cudaMemoryTypeHost) {   // pinned by the caller (cudaMallocHost / its own registration)
    cudaPointerAttributes at2;
    if (cudaPointerGetAttributes(&at2, (const char*)ptr + bytes - 1) == cudaSuccess && at2.type == cudaMemoryTypeHost) return true;
  }
  cudaGetLastError();
  bool overlapped = false;
  for (size_t i = 0; i < h->pins.size();) {
    if (h->pins[i].first < hi && lo < h->pins[i].second) {
      if (!overlapped) cudaDeviceSynchronize();          // nothing may still be reading through the old registration
      overlapped = true;
      lo = std::min(lo, h->pins[i].first); hi = std::max(hi, h->pins[i].second);
      cudaHostUnregister((void*)h->pins[i].first);
      h->pins.erase(h->pins.begin() + i);
    } else i++;
  }
  const cudaError_t e = cudaHostRegister((void*)lo, hi - lo, cudaHostRegisterDefault);
  if (e == cudaSuccess) { h->pins.emplace_back(lo, hi); return true; }
  cudaGetLastError();
  return false;
}
}  // namespace cucd

namespace {

FrameSource make_frame_source(const cucd_handle* h, const int16_t* org, long long orgPic, int orgStride, const int16_t* rec, long long recPic,
                              int recStride, uint32_t* out, uint8_t* outPacked, const uint8_t* needed = nullptr) {
  FrameSource fs;
  fs.org = org; fs.rec = rec; fs.orgPicStride = orgPic; fs.recPicStride = recPic; fs.orgStride = orgStride; fs.recStride = recStride;
  fs.W = h->cfg.width; fs.H = h->cfg.height; fs.ctusPerRow = h->ctusPerRow; fs.ctusPerPic = h->ctusPerPic; fs.out = out; fs.outPacked = outPacked; fs.needed = needed;
  return fs;
}
FeaturePlanes make_feature_planes(const cucd_handle* h, const int16_t* org, long long orgPic, int orgStride) {
  FeaturePlanes fp;
  fp.org = org; fp.orgPicStride = orgPic; fp.orgStride = orgStride; fp.W = h->cfg.width; fp.H = h->cfg.height;
  fp.ctusPerRow = h->ctusPerRow; fp.ctusPerPic = h->ctusPerPic; fp.bitDepth = h->cfg.bit_depth;
  return fp;
}

cudaError_t launch_rmd_auto(cucd_handle* h, const FrameSource& fs, int nPics, cudaStream_t st) {
  if (h->useTensor == 1 && h->cfg.bit_depth == 8) {   // kind::i8: samples are bytes
    // one scratch per handle: sized for max_pictures at creation (cucd_dev_rmd_frames may ask for more); a launch on another stream
    // than the previous one waits until that one has read it
    cudaError_t e = h->dTc2Prep.reserve(rmd_tc2_prep_bytes(nPics * h->ctusPerPic));
    if (e == cudaSuccess) e = cudaStreamWaitEvent(st, h->evTc2Prep, 0);
    if (e == cudaSuccess)
      e = launch_rmd_frames_tc2(fs, nPics, h->cfg.strong_intra_smoothing, h->dTc2Tables.p, h->dTc2Tables.p + tc2::kWinTableBytes, h->dHadamard.p,
                                h->dTc2Prep.p, st, &h->launches);
    if (e == cudaSuccess) e = cudaEventRecord(h->evTc2Prep, st);
    return e;
  }
  if (h->useTensor >= 1)      // 9/10-bit content (or path 2: any bit depth): half-precision operands, fp32 accumulators (exact integers)
    return launch_rmd_frames_tc3(fs, nPics, h->cfg.bit_depth, h->cfg.strong_intra_smoothing, h->dTc3Tables.p, h->dTc3Tables.p + tc3::kWinTableBytes16,
                                 h->dTc3Tables.p + tc3::kWinTableBytes16 + tc3::kN4TableBytes16, st, &h->launches);
  return launch_rmd_frames(fs, nPics, h->cfg.bit_depth, h->cfg.strong_intra_smoothing, st, &h->launches);
}

// planes the frame kernels read with 128-bit loads
bool plane_ok(const void* p, long long picStride, int stride, int width) {
  return ((uintptr_t)p & 15) == 0 && (stride & 7) == 0 && (picStride & 7) == 0 && stride >= width;
}

// the 15 x nPics TCM fits (TEncSlice.cpp:291-392) of one batch on the handle's worker pool: histograms -> Yc -> integer thresholds
void fit_batch(cucd_handle* h, int nPics, const uint32_t* hist, int32_t* thr, double* yc /*nPics*16*/) {
  const int nBlocks = (h->cfg.width / 4) * (h->cfg.height / 4);
  h->pool.run(nPics * 15, [=](int i) {
    const int p = i / 15, f = 1 + i % 15;
    const double y = tcm_fit_one(hist + ((size_t)p * kHistFreqs + f) * kHistBins, nBlocks);
    yc[(size_t)p * 16 + f] = y;
    thr[p * kHistFreqs + f] = (int32_t)(y * 8.0);
  });
  for (int p = 0; p < nPics; p++) { thr[p * kHistFreqs] = 0; yc[(size_t)p * 16] = 0.0; }
}

}  // namespace

extern "C" {

int cucd_abi_version(void) { return CUCD_ABI_VERSION; }

uint32_t cucd_packed_cost(const uint8_t* t, int pu, int mode) {
  if (pu < CUCD_PACKED_WIDE_PUS) return reinterpret_cast<const uint32_t*>(t)[pu * 35 + mode];
  if (pu < CUCD_PACKED_WIDE_PUS + CUCD_PACKED_U16_PUS) {
    const uint16_t v = reinterpret_cast<const uint16_t*>(t + CUCD_PACKED_U16_OFFSET)[(pu - CUCD_PACKED_WIDE_PUS) * 35 + mode];
    return v >= 0xFFFEu ? 0xFFFF0000u | v : (uint32_t)v;      /* 0xFFFF / 0xFFFE -> CUCD_COST_NOT_INSIDE / CUCD_COST_PRUNED */
  }
  const size_t bit = (size_t)((pu - CUCD_PACKED_WIDE_PUS - CUCD_PACKED_U16_PUS) * 35 + mode) * 13;
  const uint8_t* b = t + CUCD_PACKED_B13_OFFSET + (bit >> 3);
  const uint32_t w = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((bit & 7) > 3 ? (uint32_t)b[2] << 16 : 0u);   // 13 bits span 2 or 3 bytes
  const uint32_t v = (w >> (bit & 7)) & 0x1FFFu;
  return v >= 0x1FFEu ? 0xFFFFE000u | v : v;
}
void cucd_unpack_costs(const uint8_t* t, uint32_t* cost) {
  memcpy(cost, t, CUCD_PACKED_U16_OFFSET);
  const uint16_t* u = reinterpret_cast<const uint16_t*>(t + CUCD_PACKED_U16_OFFSET);
  uint32_t* o = cost + CUCD_PACKED_WIDE_PUS * 35;
  for (int i = 0; i < CUCD_PACKED_U16_PUS * 35; i++) o[i] = u[i] >= 0xFFFEu ? 0xFFFF0000u | u[i] : (uint32_t)u[i];
  o += CUCD_PACKED_U16_PUS * 35;
  const uint8_t* b = t + CUCD_PACKED_B13_OFFSET;
  // 8 values = 13 bytes: walk the stream with a 64-bit window
  uint64_t acc = 0; int have = 0; size_t pos = 0;
  for (int i = 0; i < 256 * 35; i++) {
    while (have < 13) { acc |= (uint64_t)b[pos++] << have; have += 8; }
    const uint32_t v = (uint32_t)(acc & 0x1FFFu);
    acc >>= 13; have -= 13;
    o[i] = v >= 0x1FFEu ? 0xFFFFE000u | v : v;
  }
}

const char* cucd_last_error(const cucd_handle* h) { return h ? h->err.c_str() : g_createError.c_str(); }
long long cucd_launch_count(const cucd_handle* h) { return h ? h->launchTotal + h->launches : 0; }

int cucd_create(const cucd_config* cfg, cucd_handle** out) {
  if (!cfg || !out) return fail(nullptr, CUCD_ERR_INVALID, "cucd_create: null argument");
  *out = nullptr;
  if (cfg->ctu_size != 64 || cfg->max_depth != 4) return fail(nullptr, CUCD_ERR_UNSUPPORTED, "cucd_create: only CTU 64 / depth 4 is built");
  if (cfg->bit_depth < 8 || cfg->bit_depth > 10) return fail(nullptr, CUCD_ERR_UNSUPPORTED, "cucd_create: bit depth must be 8..10");
  if (cfg->width < 8 || cfg->height < 8 || (cfg->width & 7) || (cfg->height & 7)) return fail(nullptr, CUCD_ERR_INVALID, "cucd_create: width/height must be multiples of 8");
  if (cfg->max_pictures < 1) return fail(nullptr, CUCD_ERR_INVALID, "cucd_create: max_pictures < 1");
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev <= 0) return fail(nullptr, CUCD_ERR_NO_DEVICE, std::string("cucd_create: no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU path");
  if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, CUCD_ERR_INVALID, "cucd_create: bad device ordinal");
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, cfg->device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaGetDeviceProperties");
  if (prop.major != 10) return fail(nullptr, CUCD_ERR_NO_DEVICE, "cucd_create: kernels are built for sm_100a only, device is sm_" + std::to_string(prop.major * 10 + prop.minor));
  if ((e = cudaSetDevice(cfg->device)) != cudaSuccess) return cuda_fail(nullptr, e, "cudaSetDevice");
  // per-device function attributes (> 48 KB of dynamic shared memory): once per handle, so every device a process uses is configured
  if ((e = configure_rmd_kernels()) != cudaSuccess || (e = configure_rmd_tc2_kernels()) != cudaSuccess || (e = configure_rmd_tc3_kernels()) != cudaSuccess) return cuda_fail(nullptr, e, "cudaFuncSetAttribute");

  cucd_handle* h = new cucd_handle;
  h->cfg = *cfg;
  h->ctusPerRow = (cfg->width + 63) / 64; h->ctusPerCol = (cfg->height + 63) / 64; h->ctusPerPic = h->ctusPerRow * h->ctusPerCol;
  h->pitch = (cfg->width + 63) & ~63;
  h->planeSamples = (size_t)h->pitch * cfg->height;
  // TCM fits of a 16-picture step are ~4 ms of CPU work; a handful of threads hide them behind the RMD kernel
  const int hostThreads = cfg->host_threads > 0 ? cfg->host_threads : (int)std::min(8u, std::max(1u, std::thread::hardware_concurrency()));
  h->pool.start(hostThreads);
  for (int d = 0; d < 4; d++) h->cuCount[d] = (size_t)(cfg->width / (64 >> d)) * (cfg->height / (64 >> d));
  const size_t P = (size_t)cfg->max_pictures;
  int prioLow = 0, prioHigh = 0;
  cudaDeviceGetStreamPriorityRange(&prioLow, &prioHigh);
  bool ok = cudaStreamCreateWithFlags(&h->sMain, cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithPriority(&h->sFeat, cudaStreamNonBlocking, prioHigh) == cudaSuccess &&   // small feature kernels go ahead of queued RMD blocks
            cudaStreamCreateWithFlags(&h->sGrp[0], cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&h->sGrp[1], cudaStreamNonBlocking) == cudaSuccess &&
            cudaStreamCreateWithFlags(&h->sUp, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&h->evUp, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; i < cucd_handle::kGroups; i++)
    ok = ok && cudaEventCreateWithFlags(&h->evUpG[i], cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&h->evRmdG[i], cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreate(&h->evK0) == cudaSuccess && cudaEventCreate(&h->evK1) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->evMask, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->evTc2Prep, cudaEventDisableTiming) == cudaSuccess;
  if (cfg->bit_depth == 8) ok = ok && h->dTc2Prep.reserve(rmd_tc2_prep_bytes((int)P * h->ctusPerPic)) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->evDevUp, cudaEventDisableTiming) == cudaSuccess && cudaEventCreateWithFlags(&h->evDevDone, cudaEventDisableTiming) == cudaSuccess;
  for (int i = 0; i < cucd_handle::kTimeRing; i++) ok = ok && cudaEventCreate(&h->evRmd0[i]) == cudaSuccess && cudaEventCreate(&h->evRmd1[i]) == cudaSuccess;
  for (FrameSlot& s : h->slots) {
    ok = ok && cudaEventCreateWithFlags(&s.evHist, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&s.evFork, cudaEventDisableTiming) == cudaSuccess &&
         cudaEventCreateWithFlags(&s.evJoin, cudaEventDisableTiming) == cudaSuccess;
    ok = ok && s.dHist.reserve(P * kHistFreqs * kHistBins) == cudaSuccess && s.dThr.reserve(P * kHistFreqs) == cudaSuccess;
    ok = ok && s.hHist.reserve(P * kHistFreqs * kHistBins) == cudaSuccess && s.hThr.reserve(P * kHistFreqs) == cudaSuccess;
  }
  // scratch outputs of the device-resident path for outputs the caller did not ask for; the host-buffer path sizes its own lazily
  ok = ok && h->dObf.reserve(P * (size_t)(cfg->width / 4) * (cfg->height / 4)) == cudaSuccess;
  ok = ok && h->dOutlier.reserve(P * (size_t)cfg->width * cfg->height) == cudaSuccess;
  for (int d = 0; d < 4; d++) ok = ok && h->dNum[d].reserve(P * std::max<size_t>(1, h->cuCount[d])) == cudaSuccess && h->dSum[d].reserve(P * std::max<size_t>(1, h->cuCount[d])) == cudaSuccess;
  ok = ok && h->dCtuHad.reserve(P * h->ctusPerPic) == cudaSuccess;
  ok = ok && h->dHadamard.reserve(16384) == cudaSuccess && launch_hadamard_operands(h->dHadamard.p, h->sMain) == cudaSuccess &&
       cudaStreamSynchronize(h->sMain) == cudaSuccess;
  if (ok) {
    std::vector<uint8_t> tab(tc2::kWinTableBytes + tc2::kN4TableBytes);
    tc2::fill_win_tables(tab.data()); tc2::fill_n4_tables(tab.data() + tc2::kWinTableBytes);
    ok = h->dTc2Tables.reserve(tab.size()) == cudaSuccess && cudaMemcpy(h->dTc2Tables.p, tab.data(), tab.size(), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  if (ok) {
    std::vector<uint8_t> tab(tc3::kWinTableBytes16 + tc3::kN4TableBytes16 + tc3::kHadBytes16);
    tc3::fill_win_tables16(tab.data()); tc3::fill_n4_tables16(tab.data() + tc3::kWinTableBytes16);
    tc3::fill_had_tables16(tab.data() + tc3::kWinTableBytes16 + tc3::kN4TableBytes16);
    ok = h->dTc3Tables.reserve(tab.size()) == cudaSuccess && cudaMemcpy(h->dTc3Tables.p, tab.data(), tab.size(), cudaMemcpyHostToDevice) == cudaSuccess;
  }
  h->useTensor = 1;
  { const char* ev = getenv("CUCD_RMD_PATH"); if (ev && !strcmp(ev, "alu")) h->useTensor = 0; }
  if (!ok) {
    const std::string msg = std::string("cucd_create: allocation failed: ") + cudaGetErrorString(cudaGetLastError());
    cucd_destroy(h);
    return fail(nullptr, CUCD_ERR_NOMEM, msg);
  }
  *out = h;
  return CUCD_OK;
}

int cucd_destroy(cucd_handle* h) {
  if (!h) return CUCD_OK;
  cudaSetDevice(h->cfg.device);
  cudaDeviceSynchronize();
  h->pool.stop();
  for (const auto& r : h->pins) cudaHostUnregister((void*)r.first);
  h->dOrg.release(); h->dRec.release(); h->dOrg8.release(); h->dRec8.release(); h->dObf.release(); h->dOutlier.release(); h->dObf8.release(); h->dOutlier8.release();
  h->dCost.release(); h->dCostPacked.release();
  for (FrameSlot& s : h->slots) {
    s.dHist.release(); s.hHist.release(); s.dThr.release(); s.hThr.release();
    if (s.evHist) cudaEventDestroy(s.evHist);
    if (s.evFork) cudaEventDestroy(s.evFork);
    if (s.evJoin) cudaEventDestroy(s.evJoin);
  }
  for (int d = 0; d < 4; d++) { h->dNum[d].release(); h->dSum[d].release(); }
  h->dCtuHad.release(); h->dHadamard.release(); h->dTc2Tables.release(); h->dTc2Prep.release();
  if (h->evTc2Prep) cudaEventDestroy(h->evTc2Prep);
  h->bOut.release(); h->bStage.release(); h->hStage.release(); h->hStageOut.release(); h->hScratch.release();
  for (auto& r : h->refs) r.buf.release();
  h->dCur.release(); h->dRefPtr.release(); h->dRefStride.release();
  for (auto& r : h->refCb) r.buf.release();
  for (auto& r : h->refCr) r.buf.release();
  h->dCurC.release(); h->dRefPtrC.release(); h->dRefStrideC.release();
  for (int i = 0; i < cucd_handle::kTimeRing; i++) { if (h->evRmd0[i]) cudaEventDestroy(h->evRmd0[i]); if (h->evRmd1[i]) cudaEventDestroy(h->evRmd1[i]); }
  for (int i = 0; i < cucd_handle::kGroups; i++) { if (h->evUpG[i]) cudaEventDestroy(h->evUpG[i]); if (h->evRmdG[i]) cudaEventDestroy(h->evRmdG[i]); }
  h->hDevScratch.release(); h->dDevStage.release();
  h->hSearch.release(); h->dSearch.release();
  if (h->evDevUp) cudaEventDestroy(h->evDevUp);
  if (h->evDevDone) cudaEventDestroy(h->evDevDone);
  h->dNeeded.release();
  if (h->evMask) cudaEventDestroy(h->evMask);
  if (h->evDirect) cudaEventDestroy(h->evDirect);
  if (h->evK0) cudaEventDestroy(h->evK0);
  if (h->evK1) cudaEventDestroy(h->evK1);
  if (h->sUp) cudaStreamDestroy(h->sUp);
  if (h->evUp) cudaEventDestroy(h->evUp);
  for (int i = 0; i < 2; i++) if (h->sGrp[i]) cudaStreamDestroy(h->sGrp[i]);
  if (h->sMain) cudaStreamDestroy(h->sMain);
  if (h->sFeat) cudaStreamDestroy(h->sFeat);
  delete h;
  return CUCD_OK;
}

int cucd_pin_host_buffer(cucd_handle* h, const void* ptr, size_t bytes) {
  if (!h || !ptr || !bytes) return fail(h, CUCD_ERR_INVALID, "cucd_pin_host_buffer: bad argument");
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  if (!pin_host_range(h, ptr, bytes)) return fail(h, CUCD_ERR_CUDA, "cucd_pin_host_buffer: cudaHostRegister refused the range");
  return CUCD_OK;
}
int cucd_unpin_host_buffer(cucd_handle* h, const void* ptr) {
  if (!h || !ptr) return fail(h, CUCD_ERR_INVALID, "cucd_unpin_host_buffer: bad argument");
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  CK(cudaDeviceSynchronize());
  for (size_t i = 0; i < h->pins.size(); i++)
    if (h->pins[i].first <= (uintptr_t)ptr && (uintptr_t)ptr < h->pins[i].second) {
      cudaHostUnregister((void*)h->pins[i].first);
      h->pins.erase(h->pins.begin() + i);
      return CUCD_OK;
    }
  return fail(h, CUCD_ERR_INVALID, "cucd_unpin_host_buffer: not a range this handle pinned");
}

int cucd_set_decision_switches(cucd_handle* h, int enable, const uint8_t skip2Nx2N[4], const uint8_t terminateCU[4]) {
  if (!h || (enable && (!skip2Nx2N || !terminateCU))) return fail(h, CUCD_ERR_INVALID, "cucd_set_decision_switches: bad argument");
  LOCK(h);
  if (h->begun != h->ended) return fail(h, CUCD_ERR_INVALID, "cucd_set_decision_switches: a cucd_dev_frames_begin batch is still in flight");
  h->prune = enable != 0;
  for (int d = 0; d < 4; d++) { h->sw.skip2Nx2N[d] = enable && skip2Nx2N[d] ? 1 : 0; h->sw.terminateCU[d] = enable && terminateCU[d] ? 1 : 0; }
  return CUCD_OK;
}

int cucd_set_rmd_path(cucd_handle* h, int path) {
  if (!h) return CUCD_ERR_INVALID;
  LOCK(h);
  if (path < 0 || path > 2) return fail(h, CUCD_ERR_INVALID, "cucd_set_rmd_path: path must be 0 (integer ALU), 1 (tensor cores) or 2 (half-precision tensor-core kernel at any bit depth)");
  h->useTensor = path;
  return CUCD_OK;
}

int cucd_rmd_kernel_time(cucd_handle* h, int nCalls, float* avg_ms) {
  if (!h || !avg_ms || nCalls < 1) return fail(h, CUCD_ERR_INVALID, "cucd_rmd_kernel_time: bad argument");
  LOCK(h);
  const int n = (int)std::min<long long>(std::min<long long>(nCalls, h->rmdCalls), cucd_handle::kTimeRing);
  if (n < 1) return fail(h, CUCD_ERR_INVALID, "cucd_rmd_kernel_time: no timed call yet");
  double sum = 0;
  for (int i = 0; i < n; i++) {
    const int slot = (int)((h->rmdCalls - 1 - i) % cucd_handle::kTimeRing);
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, h->evRmd0[slot], h->evRmd1[slot]));
    sum += ms;
  }
  *avg_ms = (float)(sum / n);
  return n;
}

int cucd_last_kernel_time(cucd_handle* h, float* ms) {
  if (!h || !ms) return fail(h, CUCD_ERR_INVALID, "cucd_last_kernel_time: bad argument");
  LOCK(h);
  if (!h->kTimed) return fail(h, CUCD_ERR_INVALID, "cucd_last_kernel_time: the last batch call was not timed (there was none, or it was small enough for the zero-copy path)");
  CK(cudaEventElapsedTime(ms, h->evK0, h->evK1));
  return CUCD_OK;
}

int cucd_tcm_fit(const uint32_t* hist, int nBlocks, double* yc, int32_t* thr) {
  if (!hist || !yc || !thr || nBlocks <= 0) return CUCD_ERR_INVALID;
  tcm_fit_picture(hist, nBlocks, yc, thr);
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// device-resident entry points
// ------------------------------------------------------------------------------------------------
int cucd_dev_rmd_frames(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                        const int16_t* d_rec, long long recPicStride, int recStride, uint32_t* d_rmd_cost) {
  if (!h || nPics < 1 || !d_org || !d_rec || !d_rmd_cost) return fail(h, CUCD_ERR_INVALID, "cucd_dev_rmd_frames: bad argument");
  LOCK(h);
  if (!plane_ok(d_org, orgPicStride, orgStride, h->cfg.width) || !plane_ok(d_rec, recPicStride, recStride, h->cfg.width))
    return fail(h, CUCD_ERR_INVALID, "cucd_dev_rmd_frames: source and reconstruction planes must be 16-byte aligned with strides >= width and multiples of 8");
  CK(cudaSetDevice(h->cfg.device));
  const FrameSource fs = make_frame_source(h, d_org, orgPicStride, orgStride, d_rec, recPicStride, recStride, d_rmd_cost, nullptr);
  CK(launch_rmd_auto(h, fs, nPics, (cudaStream_t)stream));
  flush_launches(h);
  return CUCD_OK;
}

int cucd_dev_feature_hist(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride, uint32_t* d_hist) {
  if (!h || nPics < 1 || !d_org || !d_hist) return fail(h, CUCD_ERR_INVALID, "cucd_dev_feature_hist: bad argument");
  LOCK(h);
  if ((orgStride & 3) || (orgPicStride & 3) || ((uintptr_t)d_org & 7) || orgStride < h->cfg.width) return fail(h, CUCD_ERR_INVALID, "cucd_dev_feature_hist: source plane must be 8-byte aligned with strides >= width and multiples of 4");
  CK(cudaSetDevice(h->cfg.device));
  CK(launch_feature_hist(make_feature_planes(h, d_org, orgPicStride, orgStride), nPics, d_hist, (cudaStream_t)stream, &h->launches));
  flush_launches(h);
  return CUCD_OK;
}

int cucd_dev_feature_obf(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                         const int32_t* d_thr, int16_t* d_obf, int16_t* d_outlier, int32_t* const d_num_obf[4],
                         int32_t* const d_n_outlier[4], int32_t* d_ctu_src_had) {
  if (!h || nPics < 1 || !d_org || !d_thr || !d_obf || !d_outlier || !d_num_obf || !d_n_outlier) return fail(h, CUCD_ERR_INVALID, "cucd_dev_feature_obf: bad argument");
  LOCK(h);
  if (!plane_ok(d_org, orgPicStride, orgStride, h->cfg.width)) return fail(h, CUCD_ERR_INVALID, "cucd_dev_feature_obf: source plane must be 16-byte aligned with strides >= width and multiples of 8");
  CK(cudaSetDevice(h->cfg.device));
  const FeaturePlanes fp = make_feature_planes(h, d_org, orgPicStride, orgStride);
  FeatureOut fo;
  fo.obf = d_obf; fo.obfPicStride = (long long)(h->cfg.width / 4) * (h->cfg.height / 4);
  fo.outlier = d_outlier; fo.outlierPicStride = (long long)h->cfg.width * h->cfg.height;
  fo.obf8 = nullptr; fo.outlier8 = nullptr;
  for (int d = 0; d < 4; d++) {
    if (!d_num_obf[d] || !d_n_outlier[d]) return fail(h, CUCD_ERR_INVALID, "cucd_dev_feature_obf: null per-depth output");
    fo.numObf[d] = d_num_obf[d]; fo.nOutlier[d] = d_n_outlier[d]; fo.cuPicStride[d] = (long long)h->cuCount[d];
  }
  CK(launch_feature_obf(fp, nPics, d_thr, fo, (cudaStream_t)stream, &h->launches));
  if (d_ctu_src_had) CK(launch_ctu_src_had(fp, nPics, d_ctu_src_had, (cudaStream_t)stream, &h->launches));
  flush_launches(h);
  return CUCD_OK;
}

int cucd_dev_frames_begin(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                          const int16_t* d_rec, long long recPicStride, int recStride, const cucd_dev_out* out, double* yc_host) {
  if (!h || nPics < 1 || nPics > h->cfg.max_pictures || !d_org || !out) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames: bad argument (nPics must be <= max_pictures)");
  LOCK(h);
  if (!plane_ok(d_org, orgPicStride, orgStride, h->cfg.width)) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames: source plane must be 16-byte aligned with strides >= width and multiples of 8");
  if ((out->rmd_cost != nullptr) != (d_rec != nullptr)) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames: d_rec and rmd_cost go together");
  if (d_rec && !plane_ok(d_rec, recPicStride, recStride, h->cfg.width)) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames: reconstruction plane must be 16-byte aligned with strides >= width and multiples of 8");
  if (h->begun - h->ended >= 2) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames_begin: two batches are already in flight - call cucd_dev_frames_end first");
  CK(cudaSetDevice(h->cfg.device));
  FrameSlot& s = h->slots[h->begun & 1];
  cudaStream_t st = (cudaStream_t)stream;
  s.st = st; s.nPics = nPics; s.out = *out; s.ycHost = yc_host;
  s.wantFeat = out->obf || out->outlier || out->ctu_src_had || yc_host || out->num_obf[0] || out->num_obf[1] || out->num_obf[2] || out->num_obf[3];
  // fork-aware mode: the RMD enumeration depends on Num_OBF, so the feature path runs first and the RMD launch moves to _end
  s.pruned = h->prune && d_rec;
  if (s.pruned) { s.wantFeat = true; s.rec = d_rec; s.recPicStride = recPicStride; s.recStride = recStride; }
  s.fp = make_feature_planes(h, d_org, orgPicStride, orgStride);
  // The feature path (two small streaming kernels around a host fit) runs on the library's high-priority stream beside the RMD
  // kernel instead of in front of / behind it: fork from the caller's stream here, join in cucd_dev_frames_end.  Its CTAs slip in
  // as RMD CTAs retire, so a step costs about the RMD launch alone.
  s.sf = st;
  if (s.wantFeat && d_rec) {
    s.sf = h->sFeat;
    CK(cudaEventRecord(s.evFork, st));
    CK(cudaStreamWaitEvent(s.sf, s.evFork, 0));
  }
  if (s.wantFeat) {
    CK(launch_feature_hist(s.fp, nPics, s.dHist.p, s.sf, &h->launches));
    CK(cudaMemcpyAsync(s.hHist.p, s.dHist.p, (size_t)nPics * kHistFreqs * kHistBins * sizeof(uint32_t), cudaMemcpyDeviceToHost, s.sf));
    CK(cudaEventRecord(s.evHist, s.sf));
  }
  if (d_rec && !s.pruned) {
    const FrameSource fs = make_frame_source(h, d_org, orgPicStride, orgStride, d_rec, recPicStride, recStride, out->rmd_cost, nullptr);
    const int slot = (int)(h->rmdCalls % cucd_handle::kTimeRing);
    CK(cudaEventRecord(h->evRmd0[slot], st));
    CK(launch_rmd_auto(h, fs, nPics, st));
    CK(cudaEventRecord(h->evRmd1[slot], st));
    h->rmdCalls++;
  }
  s.pending = true;
  h->begun++;
  flush_launches(h);
  return CUCD_OK;
}

int cucd_dev_frames_end(cucd_handle* h) {
  if (!h) return CUCD_ERR_INVALID;
  LOCK(h);
  if (h->begun == h->ended) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames_end: no batch in flight");
  CK(cudaSetDevice(h->cfg.device));
  FrameSlot& s = h->slots[h->ended & 1];
  h->ended++;
  s.pending = false;
  if (!s.wantFeat) return CUCD_OK;
  const int W = h->cfg.width, H = h->cfg.height, nPics = s.nPics;
  CK(cudaEventSynchronize(s.evHist));      // an RMD kernel keeps the GPU busy while the host fits
  std::vector<double> yc((size_t)nPics * 16, 0.0);
  fit_batch(h, nPics, s.hHist.p, s.hThr.p, yc.data());
  if (s.ycHost) memcpy(s.ycHost, yc.data(), yc.size() * sizeof(double));
  CK(cudaMemcpyAsync(s.dThr.p, s.hThr.p, (size_t)nPics * kHistFreqs * sizeof(int32_t), cudaMemcpyHostToDevice, s.sf));
  FeatureOut fo;
  fo.obf = s.out.obf ? s.out.obf : h->dObf.p; fo.obfPicStride = (long long)(W / 4) * (H / 4);
  fo.outlier = s.out.outlier ? s.out.outlier : h->dOutlier.p; fo.outlierPicStride = (long long)W * H;
  fo.obf8 = nullptr; fo.outlier8 = nullptr;
  for (int d = 0; d < 4; d++) {
    fo.numObf[d] = s.out.num_obf[d] ? s.out.num_obf[d] : h->dNum[d].p;
    fo.nOutlier[d] = s.out.n_outlier[d] ? s.out.n_outlier[d] : h->dSum[d].p;
    fo.cuPicStride[d] = (long long)h->cuCount[d];
  }
  CK(launch_feature_obf(s.fp, nPics, s.dThr.p, fo, s.sf, &h->launches));
  if (s.pruned) {
    CK(h->dNeeded.reserve((size_t)h->cfg.max_pictures * h->ctusPerPic * kPusPerCtu));
    CK(launch_prune_mask(s.fp, nPics, fo, h->sw, h->dNeeded.p, s.sf, &h->launches));
  }
  if (s.out.ctu_src_had) CK(launch_ctu_src_had(s.fp, nPics, s.out.ctu_src_had, s.sf, &h->launches));
  if (s.sf != s.st) {
    CK(cudaEventRecord(s.evJoin, s.sf));
    CK(cudaStreamWaitEvent(s.st, s.evJoin, 0));
  }
  if (s.pruned) {
    const FrameSource fs = make_frame_source(h, s.fp.org, s.fp.orgPicStride, s.fp.orgStride, s.rec, s.recPicStride, s.recStride, s.out.rmd_cost, nullptr, h->dNeeded.p);
    const int slot = (int)(h->rmdCalls % cucd_handle::kTimeRing);
    CK(cudaEventRecord(h->evRmd0[slot], s.st));
    CK(launch_rmd_auto(h, fs, nPics, s.st));
    CK(cudaEventRecord(h->evRmd1[slot], s.st));
    h->rmdCalls++;
  }
  flush_launches(h);
  return CUCD_OK;
}

int cucd_dev_frames(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                    const int16_t* d_rec, long long recPicStride, int recStride, const cucd_dev_out* out, double* yc_host) {
  if (!h) return CUCD_ERR_INVALID;
  LOCK(h);
  if (h->begun != h->ended) return fail(h, CUCD_ERR_INVALID, "cucd_dev_frames: a cucd_dev_frames_begin batch is still in flight");
  const int rc = cucd_dev_frames_begin(h, stream, nPics, d_org, orgPicStride, orgStride, d_rec, recPicStride, recStride, out, yc_host);
  return rc != CUCD_OK ? rc : cucd_dev_frames_end(h);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// S1/S4 (+ replay S2) with host buffers
// ------------------------------------------------------------------------------------------------
template <class Pel>
static int frames_group(cucd_handle* h, int nPics, const Pel* const* orgY, int strideY, const Pel* const* recY, int strideRec, cucd_frame_out* outs) {
  constexpr bool kBytes = sizeof(Pel) == 1;
  const int W = h->cfg.width, H = h->cfg.height;
  // CUCD_TRACE=1: host-side timeline of the call on stderr (development aid)
  static const bool trace = getenv("CUCD_TRACE") != nullptr;
  const auto t0 = std::chrono::steady_clock::now();
  auto stamp = [&](const char* what) {
    if (trace) fprintf(stderr, "[cucd] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
  };
  bool wantRmd = false, wantWide = false, wantPacked = false, wantObf16 = false, wantObf8 = false, wantOutl16 = false, wantOutl8 = false;
  for (int p = 0; p < nPics; p++) {
    const cucd_frame_out& o = outs[p];
    if (recY) { wantWide = wantWide || o.rmd_cost; wantPacked = wantPacked || o.rmd_cost_packed; }
    wantObf16 = wantObf16 || o.obf; wantObf8 = wantObf8 || o.obf_u8; wantOutl16 = wantOutl16 || o.outlier; wantOutl8 = wantOutl8 || o.outlier_u8;
  }
  wantRmd = wantWide || wantPacked;
  const size_t perPic = (size_t)h->ctusPerPic * kPusPerCtu * kNumModes, perPicPacked = (size_t)h->ctusPerPic * CUCD_PACKED_CTU_BYTES;
  const size_t obfPic = (size_t)(W / 4) * (H / 4), outlPic = (size_t)W * H, P = (size_t)h->cfg.max_pictures;
  // device buffers of this call's outputs, sized on first use for max_pictures
  CK(h->dOrg.reserve(P * h->planeSamples));
  if (wantRmd) CK(h->dRec.reserve(P * h->planeSamples));
  if (kBytes) { CK(h->dOrg8.reserve(P * h->planeSamples)); if (wantRmd) CK(h->dRec8.reserve(P * h->planeSamples)); }
  if (wantWide) CK(h->dCost.reserve(P * perPic));
  if (wantPacked) CK(h->dCostPacked.reserve(P * perPicPacked));
  if (wantObf8) CK(h->dObf8.reserve(P * obfPic));
  if (wantOutl8) CK(h->dOutlier8.reserve(P * outlPic));
  if (h->cfg.auto_pin_host) {
    for (int p = 0; p < nPics; p++) {
      const cucd_frame_out& o = outs[p];
      pin_host_range(h, orgY[p], ((size_t)(H - 1) * strideY + W) * sizeof(Pel));
      if (wantRmd) pin_host_range(h, recY[p], ((size_t)(H - 1) * strideRec + W) * sizeof(Pel));
      if (o.rmd_cost) pin_host_range(h, o.rmd_cost, perPic * 4);
      if (o.rmd_cost_packed) pin_host_range(h, o.rmd_cost_packed, perPicPacked);
      if (o.obf) pin_host_range(h, o.obf, obfPic * 2);
      if (o.obf_u8) pin_host_range(h, o.obf_u8, obfPic);
      if (o.outlier) pin_host_range(h, o.outlier, outlPic * 2);
      if (o.outlier_u8) pin_host_range(h, o.outlier_u8, outlPic);
    }
  }
  // ---- three-stage pipeline over sub-groups of pictures: upload (sUp) -> RMD (sGrp[0]) -> cost-table download (sGrp[1]); PCIe
  //      is full duplex, so uploads, kernels and the (dominant) downloads overlap.  The RMD kernels write the packed tables
  //      themselves.  The feature path (sFeat) needs every source plane and runs beside it. -----------------------------
  const bool pruned = h->prune && wantRmd;     // fork-aware mode: the RMD launches wait for the prune mask, i.e. for feature pass 2
  if (pruned) CK(h->dNeeded.reserve(P * h->ctusPerPic * kPusPerCtu));
  // RMD of one sub-group on sGrp[0] behind its upload (and, in fork-aware mode, behind the mask), its downloads on sGrp[1]
  auto rmd_group = [&](int gi, int first, int n) -> int {
    CK(cudaStreamWaitEvent(h->sGrp[0], h->evUpG[gi], 0));
    if (pruned) CK(cudaStreamWaitEvent(h->sGrp[0], h->evMask, 0));
    const FrameSource fs = make_frame_source(h, h->dOrg.p + (size_t)first * h->planeSamples, (long long)h->planeSamples, h->pitch,
                                             h->dRec.p + (size_t)first * h->planeSamples, (long long)h->planeSamples, h->pitch,
                                             wantWide ? h->dCost.p + (size_t)first * perPic : nullptr,
                                             wantPacked ? h->dCostPacked.p + (size_t)first * perPicPacked : nullptr,
                                             pruned ? h->dNeeded.p + (size_t)first * h->ctusPerPic * kPusPerCtu : nullptr);
    CK(launch_rmd_auto(h, fs, n, h->sGrp[0]));
    CK(cudaEventRecord(h->evRmdG[gi], h->sGrp[0]));
    CK(cudaStreamWaitEvent(h->sGrp[1], h->evRmdG[gi], 0));
    for (int p = first; p < first + n; p++) {
      if (outs[p].rmd_cost) CK(cudaMemcpyAsync(outs[p].rmd_cost, h->dCost.p + p * perPic, perPic * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->sGrp[1]));
      if (outs[p].rmd_cost_packed) CK(cudaMemcpyAsync(outs[p].rmd_cost_packed, h->dCostPacked.p + p * perPicPacked, perPicPacked, cudaMemcpyDeviceToHost, h->sGrp[1]));
    }
    return CUCD_OK;
  };
  static const int nGroups = [] { const char* e = getenv("CUCD_GROUPS"); const int g = e ? atoi(e) : 8; return std::min(std::max(g, 1), (int)cucd_handle::kGroups); }();
  const int grp = std::max(1, (nPics + nGroups - 1) / nGroups);
  int gi = 0;
  for (int first = 0; first < nPics; first += grp, gi++) {
    const int n = std::min(grp, nPics - first);
    for (int p = first; p < first + n; p++) {
      void* dOrg = kBytes ? (void*)(h->dOrg8.p + (size_t)p * h->planeSamples) : (void*)(h->dOrg.p + (size_t)p * h->planeSamples);
      CK(cudaMemcpy2DAsync(dOrg, (size_t)h->pitch * sizeof(Pel), orgY[p], (size_t)strideY * sizeof(Pel), (size_t)W * sizeof(Pel), H, cudaMemcpyHostToDevice, h->sUp));
      if (wantRmd) {
        void* dRec = kBytes ? (void*)(h->dRec8.p + (size_t)p * h->planeSamples) : (void*)(h->dRec.p + (size_t)p * h->planeSamples);
        CK(cudaMemcpy2DAsync(dRec, (size_t)h->pitch * sizeof(Pel), recY[p], (size_t)strideRec * sizeof(Pel), (size_t)W * sizeof(Pel), H, cudaMemcpyHostToDevice, h->sUp));
      }
    }
    if (kBytes) {       // bytes -> HM's Pel on the device: the planes of this group are contiguous
      CK(launch_widen_u8(h->dOrg8.p + (size_t)first * h->planeSamples, h->dOrg.p + (size_t)first * h->planeSamples, (size_t)n * h->planeSamples, h->sUp, &h->launches));
      if (wantRmd) CK(launch_widen_u8(h->dRec8.p + (size_t)first * h->planeSamples, h->dRec.p + (size_t)first * h->planeSamples, (size_t)n * h->planeSamples, h->sUp, &h->launches));
    }
    CK(cudaEventRecord(h->evUpG[gi], h->sUp));
    if (wantRmd && !pruned) { const int rc = rmd_group(gi, first, n); if (rc != CUCD_OK) return rc; }
  }
  CK(cudaEventRecord(h->evUp, h->sUp));
  // ---- feature pass 1 on sFeat -----------------------------------------------------------------
  FrameSlot& s = h->slots[0];
  CK(cudaStreamWaitEvent(h->sFeat, h->evUp, 0));
  const FeaturePlanes fp = make_feature_planes(h, h->dOrg.p, (long long)h->planeSamples, h->pitch);
  CK(launch_feature_hist(fp, nPics, s.dHist.p, h->sFeat, &h->launches));
  // histograms to the host by an SM copy (pinned memory is device-visible under UVA): a cudaMemcpyAsync would wait in the
  // copy-engine queue behind the cost-table downloads and delay the TCM fit, i.e. the whole feature path
  CK(launch_copy_words(s.dHist.p, s.hHist.p, (size_t)nPics * kHistFreqs * kHistBins, h->sFeat, &h->launches));
  CK(cudaEventRecord(s.evHist, h->sFeat));
  stamp("enqueued uploads + RMD");
  // ---- host: TCM fit per picture and frequency -------------------------------------------------
  CK(cudaEventSynchronize(s.evHist));
  stamp("histograms on host");
  std::vector<double> yc((size_t)nPics * 16, 0.0);
  fit_batch(h, nPics, s.hHist.p, s.hThr.p, yc.data());
  for (int p = 0; p < nPics; p++) if (outs[p].yc) memcpy(outs[p].yc, &yc[(size_t)p * 16], 16 * sizeof(double));
  stamp("TCM fits done");
  // ---- feature pass 2 on sFeat -----------------------------------------------------------------
  CK(cudaMemcpyAsync(s.dThr.p, s.hThr.p, (size_t)nPics * kHistFreqs * sizeof(int32_t), cudaMemcpyHostToDevice, h->sFeat));
  FeatureOut fo;
  fo.obf = wantObf16 ? h->dObf.p : nullptr; fo.obfPicStride = (long long)obfPic;
  fo.outlier = wantOutl16 ? h->dOutlier.p : nullptr; fo.outlierPicStride = (long long)outlPic;
  fo.obf8 = wantObf8 ? h->dObf8.p : nullptr; fo.outlier8 = wantOutl8 ? h->dOutlier8.p : nullptr;
  for (int d = 0; d < 4; d++) { fo.numObf[d] = h->dNum[d].p; fo.nOutlier[d] = h->dSum[d].p; fo.cuPicStride[d] = (long long)h->cuCount[d]; }
  CK(launch_feature_obf(fp, nPics, s.dThr.p, fo, h->sFeat, &h->launches));
  if (pruned) {
    CK(launch_prune_mask(fp, nPics, fo, h->sw, h->dNeeded.p, h->sFeat, &h->launches));
    CK(cudaEventRecord(h->evMask, h->sFeat));
    int g2 = 0;
    for (int first = 0; first < nPics; first += grp, g2++) { const int rc = rmd_group(g2, first, std::min(grp, nPics - first)); if (rc != CUCD_OK) return rc; }
  }
  bool wantHad = false;
  for (int p = 0; p < nPics; p++) wantHad = wantHad || outs[p].ctu_src_had;
  if (wantHad) CK(launch_ctu_src_had(fp, nPics, h->dCtuHad.p, h->sFeat, &h->launches));
  for (int p = 0; p < nPics; p++) {
    const cucd_frame_out& o = outs[p];
    if (o.obf) CK(cudaMemcpyAsync(o.obf, h->dObf.p + p * obfPic, obfPic * 2, cudaMemcpyDeviceToHost, h->sFeat));
    if (o.obf_u8) CK(cudaMemcpyAsync(o.obf_u8, h->dObf8.p + p * obfPic, obfPic, cudaMemcpyDeviceToHost, h->sFeat));
    if (o.outlier) CK(cudaMemcpyAsync(o.outlier, h->dOutlier.p + p * outlPic, outlPic * 2, cudaMemcpyDeviceToHost, h->sFeat));
    if (o.outlier_u8) CK(cudaMemcpyAsync(o.outlier_u8, h->dOutlier8.p + p * outlPic, outlPic, cudaMemcpyDeviceToHost, h->sFeat));
    for (int d = 0; d < 4; d++) {
      if (!h->cuCount[d]) continue;
      if (o.num_obf[d]) CK(cudaMemcpyAsync(o.num_obf[d], h->dNum[d].p + (size_t)p * h->cuCount[d], h->cuCount[d] * 4, cudaMemcpyDeviceToHost, h->sFeat));
      if (o.n_outlier[d]) CK(cudaMemcpyAsync(o.n_outlier[d], h->dSum[d].p + (size_t)p * h->cuCount[d], h->cuCount[d] * 4, cudaMemcpyDeviceToHost, h->sFeat));
    }
    if (o.ctu_src_had) CK(cudaMemcpyAsync(o.ctu_src_had, h->dCtuHad.p + (size_t)p * h->ctusPerPic, (size_t)h->ctusPerPic * 4, cudaMemcpyDeviceToHost, h->sFeat));
  }
  stamp("enqueued pass 2 + copies");
  CK(cudaStreamSynchronize(h->sFeat));
  stamp("feature stream done");
  CK(cudaStreamSynchronize(h->sUp));
  CK(cudaStreamSynchronize(h->sGrp[0]));
  CK(cudaStreamSynchronize(h->sGrp[1]));
  stamp("RMD streams done");
  flush_launches(h);
  return CUCD_OK;
}

template <class Pel>
static int frames_any(cucd_handle* h, const char* who, int nPics, const Pel* const* orgY, int strideY, const Pel* const* recY, int strideRec, cucd_frame_out* outs) {
  if (!h || nPics < 1 || !orgY || !outs || strideY < h->cfg.width) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": bad argument");
  LOCK(h);
  if (sizeof(Pel) == 1 && h->cfg.bit_depth != 8) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": byte planes need a handle with bit_depth 8");
  if (recY && strideRec < h->cfg.width) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": bad reconstruction stride");
  if (h->begun != h->ended) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": a cucd_dev_frames_begin batch is still in flight");
  for (int p = 0; p < nPics; p++) {
    if (!orgY[p] || (recY && !recY[p])) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": null plane");
    if ((outs[p].rmd_cost || outs[p].rmd_cost_packed) && !recY) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": rmd_cost wanted but no reconstruction plane given");
  }
  CK(cudaSetDevice(h->cfg.device));
  for (int first = 0; first < nPics; first += h->cfg.max_pictures) {
    const int n = std::min(h->cfg.max_pictures, nPics - first);
    const int rc = frames_group<Pel>(h, n, orgY + first, strideY, recY ? recY + first : nullptr, strideRec, outs + first);
    if (rc != CUCD_OK) return rc;
  }
  return CUCD_OK;
}

extern "C" {

int cuCUDecide_frames(cucd_handle* h, int nPics, const int16_t* const* orgY, int strideY, const int16_t* const* recY, int strideRec,
                      cucd_frame_out* outs) {
  return frames_any<int16_t>(h, "cuCUDecide_frames", nPics, orgY, strideY, recY, strideRec, outs);
}
int cuCUDecide_frames_u8(cucd_handle* h, int nPics, const uint8_t* const* orgY, int strideY, const uint8_t* const* recY, int strideRec,
                         cucd_frame_out* outs) {
  return frames_any<uint8_t>(h, "cuCUDecide_frames_u8", nPics, orgY, strideY, recY, strideRec, outs);
}

int cuCUDecide_frame(cucd_handle* h, const int16_t* orgY, int strideY, const int16_t* recY, int strideRec, int poc, cucd_frame_out* out) {
  (void)poc;   // the train/verify/test schedule keyed on POC (tools_YS.cpp:1237-1242) is host-side state
  const int16_t* o[1] = {orgY};
  const int16_t* r[1] = {recY};
  return cuCUDecide_frames(h, 1, o, strideY, recY ? r : nullptr, strideRec, out);
}

}  // extern "C"
