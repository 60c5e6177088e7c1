// handle.h - the state behind a cucd_handle and the small host-side helpers the C ABI files share
// (capi.cu: lifecycle + frame path, capi_batch.cu: S2 / S3 / sub-pel / TU / texture entry points).
#pragma once
#include <cuda_runtime.h>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>
#include "../../include/cucudecide.h"
#include "kernels.h"

namespace cucd {

template <class T> struct DevBuf {
  T* p = nullptr; size_t n = 0;
  cudaError_t reserve(size_t count) {
    if (count <= n) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; n = 0;
    cudaError_t e = cudaMalloc(&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
};
template <class T> struct PinBuf {
  T* p = nullptr; size_t n = 0;
  cudaError_t reserve(size_t count) {
    if (count <= n) return cudaSuccess;
    if (p) cudaFreeHost(p);
    p = nullptr; n = 0;
    cudaError_t e = cudaMallocHost(&p, count * sizeof(T));
    if (e == cudaSuccess) n = count;
    return e;
  }
  void release() { if (p) cudaFreeHost(p); p = nullptr; n = 0; }
};

struct RefPlane { DevBuf<int16_t> buf; int stride = 0, marginX = 0, marginY = 0; bool set = false; };

// Persistent worker threads for the host-side TCM fits (240 independent fits per 16-picture batch).  The pool lives as
// long as the handle: spawning threads per call costs more than the fits of a small batch, and a fixed pool keeps several
// handles / ranks on one host from oversubscribing it (cucd_config.host_threads).  The calling thread takes part.
class HostPool {
 public:
  ~HostPool() { stop(); }
  void start(int threads) {
    for (int t = 1; t < threads; t++) workers_.emplace_back([this] { loop(); });
  }
  void stop() {
    { std::lock_guard<std::mutex> lk(m_); quit_ = true; }
    cvWork_.notify_all();
    for (auto& t : workers_) if (t.joinable()) t.join();
    workers_.clear();
  }
  template <class F> void run(int n, F fn) {
    if (workers_.empty() || n <= 1) { for (int i = 0; i < n; i++) fn(i); return; }
    {
      std::lock_guard<std::mutex> lk(m_);
      job_ = fn; jobN_ = n; next_.store(0); running_ = (int)workers_.size(); gen_++;
    }
    cvWork_.notify_all();
    drain();
    std::unique_lock<std::mutex> lk(m_);
    cvDone_.wait(lk, [&] { return running_ == 0; });
    job_ = nullptr;
  }

 private:
  void drain() { for (;;) { const int i = next_.fetch_add(1); if (i >= jobN_) break; job_(i); } }
  void loop() {
    uint64_t seen = 0;
    for (;;) {
      {
        std::unique_lock<std::mutex> lk(m_);
        cvWork_.wait(lk, [&] { return quit_ || gen_ != seen; });
        if (quit_) return;
        seen = gen_;
      }
      drain();
      std::lock_guard<std::mutex> lk(m_);
      if (--running_ == 0) cvDone_.notify_all();
    }
  }
  std::vector<std::thread> workers_;
  std::mutex m_;
  std::condition_variable cvWork_, cvDone_;
  std::function<void(int)> job_;
  int jobN_ = 0, running_ = 0;
  std::atomic<int> next_{0};
  uint64_t gen_ = 0;
  bool quit_ = false;
};

// one batch of the device-resident frame path between cucd_dev_frames_begin and cucd_dev_frames_end
struct FrameSlot {
  DevBuf<uint32_t> dHist; PinBuf<uint32_t> hHist;
  DevBuf<int32_t> dThr; PinBuf<int32_t> hThr;
  cudaEvent_t evHist = nullptr, evFork = nullptr, evJoin = nullptr;
  bool pending = false, wantFeat = false, pruned = false;
  const int16_t* rec = nullptr; long long recPicStride = 0; int recStride = 0;   // pruned mode: the RMD launch happens in _end
  cudaStream_t st = nullptr, sf = nullptr;
  int nPics = 0;
  FeaturePlanes fp;
  cucd_dev_out out;
  double* ycHost = nullptr;
};

}  // namespace cucd

struct cucd_handle {
  cucd_config cfg;
  std::recursive_mutex mu;                        // every entry point holds it (see include/cucudecide.h, conventions)
  int ctusPerRow = 0, ctusPerCol = 0, ctusPerPic = 0, pitch = 0;
  size_t planeSamples = 0;
  cudaStream_t sMain = nullptr, sFeat = nullptr, sGrp[2] = {nullptr, nullptr};   // sGrp: [0] RMD compute, [1] cost-table download
  cudaStream_t sUp = nullptr;                     // picture upload
  static constexpr int kGroups = 8;               // sub-groups of pictures one cuCUDecide_frames call is pipelined over
  cudaEvent_t evUp = nullptr, evUpG[kGroups] = {}, evRmdG[kGroups] = {};
  static constexpr int kTimeRing = 64;
  cudaEvent_t evRmd0[kTimeRing] = {}, evRmd1[kTimeRing] = {};
  cudaEvent_t evK0 = nullptr, evK1 = nullptr;     // around the kernels of the last batch call (cucd_last_kernel_time)
  bool kTimed = false;
  long long rmdCalls = 0;
  int launches = 0;
  long long launchTotal = 0;
  std::string err;
  cucd::HostPool pool;
  // frame path
  cucd::FrameSlot slots[2];                       // batches in flight (begin / end)
  long long begun = 0, ended = 0;
  cucd::DevBuf<int16_t> dOrg, dRec, dObf, dOutlier;
  cucd::DevBuf<uint8_t> dOrg8, dRec8;             // cuCUDecide_frames_u8: the uploaded byte planes, widened on the device
  cucd::DevBuf<uint8_t> dObf8, dOutlier8;         // byte variants of the feature planes (cucd_frame_out.obf_u8 / outlier_u8)
  cucd::DevBuf<uint32_t> dCost;
  cucd::DevBuf<uint8_t> dCostPacked;              // CUCD_PACKED_CTU_BYTES per CTU (cucd_frame_out.rmd_cost_packed)
  cucd::DevBuf<int8_t> dHadamard;                 // +-(H8 x H8), +-(blockdiag H4 x H4) operands of the tensor-core SATD
  cucd::DevBuf<uint8_t> dTc3Tables;               // half-precision weight / Hadamard operands of the 9/10-bit tensor-core path (rmd_tc3.cuh)
  cucd::DevBuf<uint8_t> dTc2Tables;               // interpolation-weight operands of the tensor-core prediction (rmd_tc2.cuh)
  cucd::DevBuf<uint8_t> dTc2Prep;                 // 8-bit content: the border pre-pass's reference arrays, rmd_tc2_prep_bytes per launch
  cudaEvent_t evTc2Prep = nullptr;                // after the last launch that read dTc2Prep: a launch on another stream waits for it
  int useTensor = 0;                              // cucd_set_rmd_path: 1 = predictions + Hadamard on tcgen05, 0 = integer ALU
  cucd::DevBuf<int32_t> dNum[4], dSum[4], dCtuHad;
  size_t cuCount[4] = {0, 0, 0, 0};
  bool prune = false; cucd::PruneSwitches sw = {};   // fork-aware enumeration (cucd_set_decision_switches)
  cucd::DevBuf<uint8_t> dNeeded;                     // [pic][ctu][341]
  cudaEvent_t evMask = nullptr;
  std::vector<std::pair<uintptr_t, uintptr_t>> pins;   // host ranges page-locked by this handle (cucd_pin_host_buffer / auto_pin_host)
  // batch entry points (capi_batch.cu): one device block for the inputs of a call, one for its outputs; pinned staging each way for
  // small calls; pinned scratch for the job records the library builds
  cucd::DevBuf<uint8_t> bStage; cucd::DevBuf<uint32_t> bOut;
  cucd::PinBuf<uint8_t> hStage, hStageOut, hScratch;
  cudaEvent_t evDirect = nullptr;                 // completion of a zero-copy ("direct") small request (capi_batch.cu BatchIo)
  std::vector<int32_t> tmpOffA, tmpOffB;
  // ME path
  std::vector<cucd::RefPlane> refs;
  bool refTableDirty = true;
  cucd::DevBuf<int16_t> dCur; int curStride = 0; bool curSet = false;
  cucd::DevBuf<const int16_t*> dRefPtr; cucd::DevBuf<int32_t> dRefStride;
  // 4:2:0 chroma of the same slots and of the current picture (cucd_set_ref/cur_picture_chroma); setting a slot's or the current
  // luma clears its chroma flag, so a slot never pairs the luma of one picture with the chroma of another
  std::vector<cucd::RefPlane> refCb, refCr;       // per slot, set together: refCb's flag, stride and margins stand for both
  bool refTableCDirty = true;
  cucd::DevBuf<const int16_t*> dRefPtrC; cucd::DevBuf<int32_t> dRefStrideC;   // [2 slot + plane], [slot]
  cucd::DevBuf<int16_t> dCurC; int curStrideC = 0; bool curCSet = false;      // Cb plane, then Cr at curStrideC * (height / 2)
  // job records of the device-resident ME calls (cucd_dev_me_*): their own pinned / device blocks, guarded by events
  cucd::PinBuf<uint8_t> hDevScratch; cucd::DevBuf<uint8_t> dDevStage;
  // cucd_me_search: pinned records (cost records, sub-pel jobs, FRAC list) beside hScratch's ME jobs / tiles, and device scratch
  // (keys, completed sub-pel jobs, 49-entry tables)
  cucd::PinBuf<uint8_t> hSearch; cucd::DevBuf<uint8_t> dSearch;
  cudaEvent_t evDevUp = nullptr, evDevDone = nullptr; bool devBusy = false;
};

namespace cucd {

extern std::string g_createError;
inline int fail(cucd_handle* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_createError = msg;
  return code;
}
inline int cuda_fail(cucd_handle* h, cudaError_t e, const char* what) {
  return fail(h, CUCD_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CK(call)                                                         \
  do {                                                                   \
    cudaError_t e__ = (call);                                            \
    if (e__ != cudaSuccess) return cucd::cuda_fail(h, e__, #call);       \
  } while (0)
#define LOCK(h) std::lock_guard<std::recursive_mutex> lock__((h)->mu)

inline void flush_launches(cucd_handle* h) { h->launchTotal += h->launches; h->launches = 0; }

// page-lock [ptr, ptr + bytes) for the lifetime of the handle; false if the range could not be registered (the transfer
// then takes the pageable path, which is still correct)
bool pin_host_range(cucd_handle* h, const void* ptr, size_t bytes);

}  // namespace cucd
