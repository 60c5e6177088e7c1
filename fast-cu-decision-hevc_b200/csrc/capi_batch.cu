// capi_batch.cu - the batch entry points of the C ABI (include/cucudecide.h): S2 intra RMD batches and their coalescing queue,
// S3 integer-ME SAD surfaces, fractional-pel refinement, the intra TU coding chain, CU texture features and AQ activity.
// Size-class bucketing of the requests and tiling of the ME search windows happen here; there is no CPU compute path.
//
// How caller buffers travel (BatchIo): every input array of a call gets a 16-byte aligned place in ONE device block and every
// output array in another.  Small calls (<= 1 MB each way: what a live encoder sends) go through the handle's pinned staging
// blocks - one copy up, one copy down, no pageable transfer.  Large calls (a picture's worth) are copied array by array straight
// from / to the caller's memory: by DMA when that memory is page-locked (cucd_pin_host_buffer, auto_pin_host, or pinned by
// the caller), through the driver's pageable path otherwise.  Arrays the library builds itself (PU / TU / ME job records) are
// written once, in size-class order, into pinned scratch.
#include <cuda_runtime.h>
#include <algorithm>
#include <chrono>
#include <cstring>
#include <deque>
#include "handle.h"
#include "rmd_tc2.cuh"
#include "me_core.cuh"

using namespace cucd;

namespace {

constexpr size_t kStageLimit = (size_t)1 << 20;
inline size_t up16(size_t v) { return (v + 15) & ~(size_t)15; }

bool host_pinned(cucd_handle* h, const void* p, size_t bytes) {
  const uintptr_t lo = (uintptr_t)p, hi = lo + bytes;
  for (const auto& r : h->pins) if (r.first <= lo && hi <= r.second) return true;
  if (h->cfg.auto_pin_host) return pin_host_range(h, p, bytes);
  cudaPointerAttributes at;
  const bool pinned = cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeHost;
  cudaGetLastError();
  return pinned;
}

// Requests of a live encoder are tiny (one PU: ~1 KB in, 140 B out; one 128 x 128 SAD tile: 64 KB out) and latency bound: two DMA
// copies, two timing events and a blocking stream wait cost several times the kernel.  Below `directLimit` bytes the kernels read
// their inputs from and write their results to page-locked HOST memory directly (zero copy over PCIe, unified addressing) and the
// call polls one event: a host memcpy each way, the launches, one cudaEventRecord.  CUCD_DIRECT_LIMIT=<bytes> (0 = off).
inline size_t direct_limit() {
  static const size_t v = [] { const char* e = getenv("CUCD_DIRECT_LIMIT"); return e ? (size_t)strtoull(e, nullptr, 10) : (size_t)96 << 10; }();
  return v;
}

struct BatchIo {
  struct Part { const void* src; void* dst; size_t bytes, off; bool pinned; };
  cucd_handle* h;
  Part in[8], out[8];
  int nIn = 0, nOut = 0;
  size_t inBytes = 0, outBytes = 0;
  bool direct = false;
  explicit BatchIo(cucd_handle* hh) : h(hh) {}
  int add_in(const void* src, size_t bytes, bool pinned = false) { in[nIn] = Part{src, nullptr, bytes, inBytes, pinned}; inBytes += up16(bytes); return nIn++; }
  int add_out(void* dst, size_t bytes) { out[nOut] = Part{nullptr, dst, dst ? bytes : 0, outBytes, false}; outBytes += up16(dst ? bytes : 0); return nOut++; }
  // device-side room for an array the kernels produce but the caller did not ask for
  int add_scratch_out(size_t bytes) { out[nOut] = Part{nullptr, nullptr, 0, outBytes, false}; outBytes += up16(bytes); return nOut++; }
  int reserve() {
    direct = inBytes + outBytes <= direct_limit() && inBytes + 256 <= kStageLimit && outBytes + 256 <= kStageLimit;
    if (direct) {
      CK(h->hStage.reserve(kStageLimit)); CK(h->hStageOut.reserve(kStageLimit));
      if (!h->evDirect) CK(cudaEventCreateWithFlags(&h->evDirect, cudaEventDisableTiming));
      return CUCD_OK;
    }
    CK(h->bStage.reserve(inBytes + 256));
    CK(h->bOut.reserve(outBytes / 4 + 64));
    return CUCD_OK;
  }
  template <class T> T* din(int i) const { return reinterpret_cast<T*>((direct ? h->hStage.p : h->bStage.p) + in[i].off); }
  template <class T> T* dout(int i) const { return reinterpret_cast<T*>((direct ? h->hStageOut.p : reinterpret_cast<uint8_t*>(h->bOut.p)) + out[i].off); }
  int upload(cudaStream_t st) {
    if (direct) {
      for (int i = 0; i < nIn; i++) if (in[i].bytes) memcpy(h->hStage.p + in[i].off, in[i].src, in[i].bytes);
      return CUCD_OK;
    }
    bool allPinned = true;
    for (int i = 0; i < nIn; i++) allPinned = allPinned && in[i].pinned;
    if (inBytes <= kStageLimit && !allPinned) {
      CK(h->hStage.reserve(kStageLimit));
      for (int i = 0; i < nIn; i++) if (in[i].bytes) memcpy(h->hStage.p + in[i].off, in[i].src, in[i].bytes);
      CK(cudaMemcpyAsync(h->bStage.p, h->hStage.p, inBytes, cudaMemcpyHostToDevice, st));
      return CUCD_OK;
    }
    for (int i = 0; i < nIn; i++) {
      if (!in[i].bytes) continue;
      if (!in[i].pinned && in[i].bytes >= (64u << 10)) host_pinned(h, in[i].src, in[i].bytes);    // registers the range when auto_pin_host is set
      CK(cudaMemcpyAsync(h->bStage.p + in[i].off, in[i].src, in[i].bytes, cudaMemcpyHostToDevice, st));
    }
    return CUCD_OK;
  }
  // enqueue the copies back, wait for the stream, hand the results to the caller
  int download(cudaStream_t st) {
    if (direct) {
      CK(cudaEventRecord(h->evDirect, st));
      cudaError_t e;
      while ((e = cudaEventQuery(h->evDirect)) == cudaErrorNotReady) { }
      CK(e);
      for (int i = 0; i < nOut; i++) if (out[i].bytes) memcpy(out[i].dst, h->hStageOut.p + out[i].off, out[i].bytes);
      return CUCD_OK;
    }
    size_t wanted = 0;
    for (int i = 0; i < nOut; i++) wanted += out[i].bytes;
    if (outBytes <= kStageLimit) {
      CK(h->hStageOut.reserve(kStageLimit));
      if (wanted) CK(cudaMemcpyAsync(h->hStageOut.p, h->bOut.p, outBytes, cudaMemcpyDeviceToHost, st));
      CK(cudaStreamSynchronize(st));
      for (int i = 0; i < nOut; i++) if (out[i].bytes) memcpy(out[i].dst, h->hStageOut.p + out[i].off, out[i].bytes);
      return CUCD_OK;
    }
    for (int i = 0; i < nOut; i++) {
      if (!out[i].bytes) continue;
      if (out[i].bytes >= (64u << 10)) host_pinned(h, out[i].dst, out[i].bytes);
      CK(cudaMemcpyAsync(out[i].dst, reinterpret_cast<uint8_t*>(h->bOut.p) + out[i].off, out[i].bytes, cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    return CUCD_OK;
  }
};

// ---- S2 core: PUs described by (size, sample offsets into `org` / `border`); the records are bucketed by size into pinned scratch ----
int rmd_batch_core(cucd_handle* h, int nPU, const cucd_pu_desc* desc, const int32_t* orgOffs, const int32_t* borderOffs, const int16_t* org, size_t orgSamples,
                   const int16_t* border, size_t borderSamples, bool inputsPinned, uint32_t* sad) {
  // counting sort by size class straight into pinned scratch
  int count[7] = {0}, first[7] = {0};
  for (int i = 0; i < nPU; i++) count[desc[i].log2_size]++;
  for (int l = 3; l <= 6; l++) first[l] = first[l - 1] + count[l - 1];
  CK(h->hScratch.reserve((size_t)nPU * sizeof(BatchPu) + 64));
  BatchPu* pus = reinterpret_cast<BatchPu*>(h->hScratch.p);
  {
    int next[7];
    for (int l = 2; l <= 6; l++) next[l] = first[l];
    for (int i = 0; i < nPU; i++) {
      BatchPu& b = pus[next[desc[i].log2_size]++];
      b.orgOff = orgOffs[i]; b.borderOff = borderOffs[i]; b.outIndex = i; b.pad = 0;
    }
  }
  BatchIo io(h);
  const int iOrg = io.add_in(org, orgSamples * 2, inputsPinned);
  const int iBrd = border == org ? iOrg : io.add_in(border, borderSamples * 2, inputsPinned);   // the queue keeps both in one arena
  const int iPus = io.add_in(pus, (size_t)nPU * sizeof(BatchPu), true);
  io.inBytes += 256;                                  // the kernels read whole 16-byte words past the last block
  const int oSad = io.add_out(sad, (size_t)nPU * kNumModes * sizeof(uint32_t));
  if (io.reserve() != CUCD_OK) return CUCD_ERR_CUDA;
  if (io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  if (!io.direct) CK(cudaEventRecord(h->evK0, h->sMain));
  for (int l = 6; l >= 2; l--) {
    if (!count[l]) continue;
    BatchSource bs;
    bs.org = io.din<int16_t>(iOrg); bs.border = io.din<int16_t>(iBrd); bs.pus = io.din<BatchPu>(iPus) + first[l]; bs.out = io.dout<uint32_t>(oSad); bs.count = count[l];
    // A handful of PUs (what a live encoder sends per request) is latency bound: the integer-ALU kernel spreads the 35 modes over its
    // warps and finishes a lone PU in a few microseconds, the tensor-core kernel walks its 19 MMA rounds whatever the row count.
    // The tensor-core kernel wins on throughput as soon as there is more than one chunk (4096 samples) of a size.
    const bool small = count[l] <= (4096 >> (2 * l));
    if (h->useTensor == 1 && h->cfg.bit_depth == 8 && !small)
      CK(launch_rmd_batch_tc2(l, bs, h->cfg.strong_intra_smoothing, h->dTc2Tables.p, h->dTc2Tables.p + tc2::kWinTableBytes, h->dHadamard.p, h->sMain, &h->launches));
    else
      CK(launch_rmd_batch(l, bs, h->cfg.bit_depth, h->cfg.strong_intra_smoothing, h->sMain, &h->launches));
  }
  if (!io.direct) { CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true; } else h->kTimed = false;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}

// offsets of back-to-back packed PUs (the layout of the public batch calls); false on a bad size or an overflowing batch
bool packed_offsets(int n, const uint8_t* log2s, int stride, int lo, int hi, std::vector<int32_t>& orgOffs, std::vector<int32_t>& brdOffs, size_t& orgN, size_t& brdN) {
  orgOffs.resize(n); brdOffs.resize(n);
  orgN = 0; brdN = 0;
  for (int i = 0; i < n; i++) {
    const int l = log2s[(size_t)i * stride];
    if (l < lo || l > hi) return false;
    orgOffs[i] = (int32_t)orgN; brdOffs[i] = (int32_t)brdN;
    orgN += (size_t)1 << (2 * l); brdN += ((size_t)4 << l) + 1;
    if (orgN > 0x7fff0000ull || brdN > 0x7fff0000ull) return false;
  }
  return true;
}

}  // namespace

extern "C" {

// ------------------------------------------------------------------------------------------------
// S2: batched RMD with caller-supplied borders
// ------------------------------------------------------------------------------------------------
int cucd_intra_rmd_batch(cucd_handle* h, int nPU, const cucd_pu_desc* desc, const int16_t* org, const int16_t* border, uint32_t* sad) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !org || !border || !sad))) return fail(h, CUCD_ERR_INVALID, "cucd_intra_rmd_batch: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  std::vector<int32_t>& orgOffs = h->tmpOffA; std::vector<int32_t>& brdOffs = h->tmpOffB;
  size_t orgN, brdN;
  if (!packed_offsets(nPU, &desc[0].log2_size, (int)sizeof(cucd_pu_desc), 2, 6, orgOffs, brdOffs, orgN, brdN))
    return fail(h, CUCD_ERR_INVALID, "cucd_intra_rmd_batch: log2_size must be 2..6 and a batch at most 2^31 samples");
  const int rc = rmd_batch_core(h, nPU, desc, orgOffs.data(), brdOffs.data(), org, orgN, border, brdN, false, sad);
  return rc;
}

// ------------------------------------------------------------------------------------------------
// S2, asynchronous and coalescing: a worker thread turns everything that is pending into one batch.
// Submitters copy their request ONCE, into the pinned arena that is currently being filled; the worker swaps arenas and
// uploads straight from the one it took.  A short batching window lets the requests of the other instances arrive: after
// a batch completes all its submitters are released together and come back within tens of microseconds.
// ------------------------------------------------------------------------------------------------
struct cucd_queue {
  struct Item { uint64_t ticket; int nPU; int firstPu; uint32_t* sad; };
  struct Arena {
    PinBuf<int16_t> samples; size_t used = 0;          // org and border blocks of every request, back to back
    std::vector<Item> items; std::vector<cucd_pu_desc> desc; std::vector<int32_t> orgOff, brdOff;
    void clear() { used = 0; items.clear(); desc.clear(); orgOff.clear(); brdOff.clear(); }
  };
  cucd_handle* h = nullptr;
  std::mutex m;
  std::condition_variable cvWork, cvDone;
  Arena arena[2];
  int fill = 0;
  uint64_t nextTicket = 1, doneUpTo = 0;
  std::deque<std::pair<uint64_t, std::pair<uint64_t, int>>> failed;   // (first ticket, (last ticket, status)) of failed batches still worth remembering
  bool stop = false;
  int windowUs = 30, lastBatchRequests = 1;
  long long requests = 0, pus = 0, batches = 0;
  std::thread worker;

  void run() {
    std::vector<uint32_t> sad;
    for (;;) {
      Arena* a;
      {
        std::unique_lock<std::mutex> lk(m);
        cvWork.wait(lk, [&] { return stop || !arena[fill].items.empty(); });
        if (arena[fill].items.empty()) return;       // stop requested and nothing left
        // batching window: the instances released by the previous batch are on their way back
        if (windowUs > 0 && !stop && (int)arena[fill].items.size() < lastBatchRequests) {
          const auto deadline = std::chrono::steady_clock::now() + std::chrono::microseconds(windowUs);
          cvWork.wait_until(lk, deadline, [&] { return stop || (int)arena[fill].items.size() >= lastBatchRequests; });
        }
        a = &arena[fill];
        fill ^= 1;
      }
      const int total = (int)a->desc.size();
      sad.resize((size_t)total * kNumModes);
      int rc = CUCD_OK;
      if (total) {
        LOCK(h);
        rc = cudaSetDevice(h->cfg.device) == cudaSuccess
               ? rmd_batch_core(h, total, a->desc.data(), a->orgOff.data(), a->brdOff.data(), a->samples.p, a->used, a->samples.p, a->used, true, sad.data())
               : CUCD_ERR_CUDA;
      }
      if (rc == CUCD_OK)
        for (const Item& it : a->items) memcpy(it.sad, sad.data() + (size_t)it.firstPu * kNumModes, (size_t)it.nPU * kNumModes * sizeof(uint32_t));
      {
        std::lock_guard<std::mutex> lk(m);
        if (rc != CUCD_OK) { failed.emplace_back(a->items.front().ticket, std::make_pair(a->items.back().ticket, rc)); if (failed.size() > 64) failed.pop_front(); }
        doneUpTo = a->items.back().ticket;
        lastBatchRequests = (int)a->items.size();
        batches++;
        a->clear();
      }
      cvDone.notify_all();
    }
  }
};

int cucd_queue_create(cucd_handle* h, cucd_queue** out) {
  if (!h || !out) return fail(h, CUCD_ERR_INVALID, "cucd_queue_create: null argument");
  cucd_queue* q = new cucd_queue;
  q->h = h;
  { const char* e = getenv("CUCD_QUEUE_WINDOW_US"); if (e) q->windowUs = std::max(0, atoi(e)); }
  q->worker = std::thread([q] { q->run(); });
  *out = q;
  return CUCD_OK;
}

int cucd_queue_destroy(cucd_queue* q) {
  if (!q) return CUCD_OK;
  { std::lock_guard<std::mutex> lk(q->m); q->stop = true; }
  q->cvWork.notify_all();
  if (q->worker.joinable()) q->worker.join();
  for (auto& a : q->arena) a.samples.release();
  delete q;
  return CUCD_OK;
}

int cucd_queue_submit(cucd_queue* q, int nPU, const cucd_pu_desc* desc, const int16_t* org, const int16_t* border, uint32_t* sad, uint64_t* ticket) {
  if (!q || !ticket || nPU < 0 || (nPU > 0 && (!desc || !org || !border || !sad))) return CUCD_ERR_INVALID;
  size_t orgN = 0, brdN = 0;
  for (int i = 0; i < nPU; i++) {
    const int l = desc[i].log2_size;
    if (l < 2 || l > 6) return CUCD_ERR_INVALID;
    orgN += (size_t)1 << (2 * l); brdN += ((size_t)4 << l) + 1;
  }
  {
    std::lock_guard<std::mutex> lk(q->m);
    if (q->stop) return CUCD_ERR_INVALID;
    cucd_queue::Arena& a = q->arena[q->fill];
    const size_t need = a.used + ((orgN + 7) & ~(size_t)7) + ((brdN + 7) & ~(size_t)7);
    if (need > 0x7fff0000ull) return CUCD_ERR_INVALID;
    if (need > a.samples.n) {                          // grow the pinned arena (rare: sizes settle after the first batches)
      PinBuf<int16_t> bigger;
      cudaSetDevice(q->h->cfg.device);
      if (bigger.reserve(std::max(need * 2, (size_t)1 << 18)) != cudaSuccess) return CUCD_ERR_NOMEM;
      if (a.used) memcpy(bigger.p, a.samples.p, a.used * 2);
      a.samples.release();
      a.samples = bigger;
    }
    // the single copy of the request: source blocks (16-byte aligned, the kernels read them with 128-bit loads), then borders
    size_t o = a.used, b = a.used + ((orgN + 7) & ~(size_t)7);
    memcpy(a.samples.p + o, org, orgN * 2);
    memcpy(a.samples.p + b, border, brdN * 2);
    const int firstPu = (int)a.desc.size();
    for (int i = 0; i < nPU; i++) {
      const int l = desc[i].log2_size;
      a.desc.push_back(desc[i]); a.orgOff.push_back((int32_t)o); a.brdOff.push_back((int32_t)b);
      o += (size_t)1 << (2 * l); b += ((size_t)4 << l) + 1;
    }
    a.used = need;
    const uint64_t t = *ticket = q->nextTicket++;
    a.items.push_back(cucd_queue::Item{t, nPU, firstPu, sad});
    q->requests++; q->pus += nPU;
  }
  q->cvWork.notify_one();
  return CUCD_OK;
}

int cucd_queue_wait(cucd_queue* q, uint64_t ticket) {
  if (!q || ticket == 0) return CUCD_ERR_INVALID;
  std::unique_lock<std::mutex> lk(q->m);
  if (ticket >= q->nextTicket) return CUCD_ERR_INVALID;
  q->cvDone.wait(lk, [&] { return q->doneUpTo >= ticket; });
  for (const auto& f : q->failed) if (ticket >= f.first && ticket <= f.second.first) return f.second.second;   // only tickets of a failed batch see its status
  return CUCD_OK;
}

int cucd_queue_stats(cucd_queue* q, long long* requests, long long* pus, long long* batches) {
  if (!q) return CUCD_ERR_INVALID;
  std::lock_guard<std::mutex> lk(q->m);
  if (requests) *requests = q->requests;
  if (pus) *pus = q->pus;
  if (batches) *batches = q->batches;
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// S3: integer ME SAD surfaces
// ------------------------------------------------------------------------------------------------
int cucd_set_ref_picture(cucd_handle* h, int ref_idx, const int16_t* recY, int stride, int marginX, int marginY) {
  if (!h || ref_idx < 0 || ref_idx >= 64 || !recY || marginX < 0 || marginY < 0 || stride < h->cfg.width + 2 * marginX)
    return fail(h, CUCD_ERR_INVALID, "cucd_set_ref_picture: bad argument");
  LOCK(h);
  // the slot's chroma belongs to the picture being replaced: unset it before anything can fail
  if ((int)h->refCb.size() > ref_idx) h->refCb[ref_idx].set = false;
  CK(cudaSetDevice(h->cfg.device));
  if ((int)h->refs.size() <= ref_idx) h->refs.resize(ref_idx + 1);
  RefPlane& r = h->refs[ref_idx];
  const int pw = h->cfg.width + 2 * marginX, ph = h->cfg.height + 2 * marginY;
  const int pitch = (pw + 7) & ~7;
  CK(r.buf.reserve((size_t)pitch * ph));
  const int16_t* first = recY - (ptrdiff_t)marginY * stride - marginX;
  if (h->cfg.auto_pin_host) pin_host_range(h, first, ((size_t)(ph - 1) * stride + pw) * 2);
  CK(cudaMemcpy2DAsync(r.buf.p, (size_t)pitch * 2, first, (size_t)stride * 2, (size_t)pw * 2, ph, cudaMemcpyHostToDevice, h->sMain));
  CK(cudaStreamSynchronize(h->sMain));
  r.stride = pitch; r.marginX = marginX; r.marginY = marginY; r.set = true;
  h->refTableDirty = true;
  return CUCD_OK;
}

int cucd_set_cur_picture(cucd_handle* h, const int16_t* orgY, int stride) {
  if (!h || !orgY || stride < h->cfg.width) return fail(h, CUCD_ERR_INVALID, "cucd_set_cur_picture: bad argument");
  LOCK(h);
  h->curCSet = false;                              // likewise the current chroma
  CK(cudaSetDevice(h->cfg.device));
  CK(h->dCur.reserve(h->planeSamples));
  if (h->cfg.auto_pin_host) pin_host_range(h, orgY, ((size_t)(h->cfg.height - 1) * stride + h->cfg.width) * 2);
  CK(cudaMemcpy2DAsync(h->dCur.p, (size_t)h->pitch * 2, orgY, (size_t)stride * 2, (size_t)h->cfg.width * 2, h->cfg.height, cudaMemcpyHostToDevice, h->sMain));
  CK(cudaStreamSynchronize(h->sMain));
  h->curStride = h->pitch; h->curSet = true;
  return CUCD_OK;
}

// the device-side table of resident reference planes changes only when a plane is (re)allocated: upload it then, not per call
static int sync_ref_table(cucd_handle* h) {
  if (!h->refTableDirty) return CUCD_OK;
  std::vector<const int16_t*> refPtr(h->refs.size(), nullptr);
  std::vector<int32_t> refStride(h->refs.size(), 0);
  for (size_t i = 0; i < h->refs.size(); i++) { refPtr[i] = h->refs[i].buf.p; refStride[i] = h->refs[i].stride; }
  CK(h->dRefPtr.reserve(std::max<size_t>(64, refPtr.size()))); CK(h->dRefStride.reserve(std::max<size_t>(64, refStride.size())));
  CK(cudaMemcpyAsync(h->dRefPtr.p, refPtr.data(), refPtr.size() * sizeof(void*), cudaMemcpyHostToDevice, h->sMain));
  CK(cudaMemcpyAsync(h->dRefStride.p, refStride.data(), refStride.size() * 4, cudaMemcpyHostToDevice, h->sMain));
  CK(cudaStreamSynchronize(h->sMain));                 // the vectors above are about to go away
  h->refTableDirty = false;
  return CUCD_OK;
}

// validate the PUs, build job + tile records into `scratch` (pinned); returns the sizes through the references
// ownBlocks: the source blocks are the caller's (cucd_me_sad_surface_src): offsets run through the packed block array
// Tile records (me_core.cuh): the dy-lane tiles of every PU first, then the dx-lane tiles; nTilesDy / nTilesO count them.
static int me_build_jobs(cucd_handle* h, int nPU, const cucd_me_desc* desc, PinBuf<uint8_t>& scratch, size_t& jobBytes, size_t& tileBytes, long long& total, long long& nTilesDy,
                         long long& nTilesO, bool ownBlocks = false, size_t* srcSamples = nullptr) {
  const int W = h->cfg.width, H = h->cfg.height;
  const int tileRows = (h->cfg.bit_depth == 8 && !ownBlocks) ? 16 : 8;     // me_sad_u8_kernel covers 32 x 16 candidates per CTA, me_sad_kernel 32 x 8
  const bool fast = !ownBlocks;                                            // caller-supplied blocks may hold signed samples: dx-lane kernel only
  total = 0; nTilesDy = 0; nTilesO = 0;
  for (int i = 0; i < nPU; i++) {
    const cucd_me_desc& d = desc[i];
    // HM's PU widths are multiples of 4 (4..64, AMP 12 / 24 / 48 included); the 8-bit kernel reads the source as 32-bit words
    if (d.w < 4 || d.h < 4 || d.w > 64 || d.h > 64 || (d.w & 3) || d.x < 0 || d.y < 0 || d.x + d.w > W || d.y + d.h > H || d.left > d.right || d.top > d.bottom ||
        d.sub_shift < 0 || d.sub_shift > 4)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: bad PU / window (width must be a multiple of 4)");
    if (d.ref_idx < 0 || d.ref_idx >= (int)h->refs.size() || !h->refs[d.ref_idx].set) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: reference picture not set");
    const RefPlane& r = h->refs[d.ref_idx];
    if (d.x + d.left < -r.marginX || d.y + d.top < -r.marginY || d.x + d.w - 1 + d.right > W - 1 + r.marginX || d.y + d.h - 1 + d.bottom > H - 1 + r.marginY)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: window leaves the padded reference picture");
    const int cols = d.right - d.left + 1, rows = d.bottom - d.top + 1;
    if (cols > kMeMaxWindow || rows > kMeMaxWindow) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: window too large");
    me_enum_tiles(cols, rows, fast && me_width_is_hm(d.w), tileRows, [&](int kind, int, int) { if (kind == kMeKindO) nTilesO++; else nTilesDy++; });
    total += (long long)cols * rows;
  }
  const long long nTiles = nTilesDy + nTilesO;
  if (nTiles > 0x7fffffffll) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: batch too large");
  jobBytes = up16((size_t)nPU * sizeof(MeJob)); tileBytes = up16((size_t)nTiles * 4);
  CK(scratch.reserve(jobBytes + 2 * tileBytes));
  MeJob* jobs = reinterpret_cast<MeJob*>(scratch.p);
  int32_t* tileJob = reinterpret_cast<int32_t*>(scratch.p + jobBytes);
  int32_t* tileIdx = reinterpret_cast<int32_t*>(scratch.p + jobBytes + tileBytes);
  long long off = 0; size_t ntDy = 0, ntO = (size_t)nTilesDy, blockOff = 0;
  for (int i = 0; i < nPU; i++) {
    const cucd_me_desc& d = desc[i];
    const RefPlane& r = h->refs[d.ref_idx];
    MeJob& j = jobs[i];
    j.curOff = ownBlocks ? (int32_t)blockOff : d.y * h->curStride + d.x;
    blockOff += (size_t)d.w * d.h;
    j.refOff = (d.y + r.marginY) * r.stride + d.x + r.marginX;
    j.refSlot = d.ref_idx; j.w = (int16_t)d.w; j.h = (int16_t)d.h;
    j.left = (int16_t)d.left; j.right = (int16_t)d.right; j.top = (int16_t)d.top; j.bottom = (int16_t)d.bottom;
    // the width-specialised xGetSAD* honour iSubShift, the generic xGetSAD (TComRdCost.cpp:465-491) does not
    const bool special = me_width_is_hm(d.w);
    j.subShift = (int16_t)(special ? d.sub_shift : 0); j.pad = 0;
    j.outOff = off;
    const int cols = d.right - d.left + 1, rows = d.bottom - d.top + 1;
    me_enum_tiles(cols, rows, fast && special, tileRows, [&](int kind, int x0, int y0) {
      size_t& nt = kind == kMeKindO ? ntO : ntDy;
      tileJob[nt] = i; tileIdx[nt] = me_tile_pack(kind, x0, y0); nt++;
    });
    off += (long long)cols * rows;
  }
  if (blockOff > 0x7fffffffull) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface_src: batch too large");
  if (srcSamples) *srcSamples = blockOff;
  return CUCD_OK;
}

static int me_sad_surface_impl(cucd_handle* h, int nPU, const cucd_me_desc* desc, const int16_t* src, uint32_t* sadOut) {
  const bool own = src != nullptr;
  if (!own && !h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  size_t jobBytes, tileBytes, srcSamples = 0; long long total, nTilesDy, nTilesO;
  const int rc = me_build_jobs(h, nPU, desc, h->hScratch, jobBytes, tileBytes, total, nTilesDy, nTilesO, own, &srcSamples);
  if (rc != CUCD_OK) return rc;
  if (sync_ref_table(h) != CUCD_OK) return CUCD_ERR_CUDA;
  BatchIo io(h);
  const int iAll = io.add_in(h->hScratch.p, jobBytes + 2 * tileBytes, true);
  const int iSrc = own ? io.add_in(src, srcSamples * sizeof(int16_t)) : -1;
  const int oSad = io.add_out(sadOut, (size_t)total * sizeof(uint32_t));
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  MePlanes mp;
  mp.cur = own ? io.din<int16_t>(iSrc) : h->dCur.p; mp.curStride = own ? 0 : h->curStride;
  mp.ref = h->dRefPtr.p; mp.refStride = h->dRefStride.p; mp.bitDepth = h->cfg.bit_depth;
  const uint8_t* dAll = io.din<uint8_t>(iAll);
  if (!io.direct) CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_me_sad(mp, reinterpret_cast<const MeJob*>(dAll), nPU, reinterpret_cast<const int32_t*>(dAll + jobBytes), reinterpret_cast<const int32_t*>(dAll + jobBytes + tileBytes),
                   (int)nTilesDy, (int)nTilesO, io.dout<uint32_t>(oSad), h->sMain, &h->launches));
  if (!io.direct) { CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true; } else h->kTimed = false;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}
int cucd_me_sad_surface(cucd_handle* h, int nPU, const cucd_me_desc* desc, uint32_t* sadOut) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !sadOut))) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  return me_sad_surface_impl(h, nPU, desc, nullptr, sadOut);
}
int cucd_me_sad_surface_src(cucd_handle* h, int nPU, const cucd_me_desc* desc, const int16_t* src, uint32_t* sadOut) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !src || !sadOut))) return fail(h, CUCD_ERR_INVALID, "cucd_me_sad_surface_src: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  return me_sad_surface_impl(h, nPU, desc, src, sadOut);
}

// Device-resident variants: the surfaces / cost tables stay in HBM (d_out), everything is enqueued on `stream` and the call does
// not wait for the GPU.  The job records travel through buffers of their own, guarded by an event, so that back-to-back calls on
// one stream pipeline and a host-buffer call in between cannot overwrite records a queued kernel still has to read.
static int dev_records_begin(cucd_handle* h, cudaStream_t st) {
  if (h->devBusy) { CK(cudaEventSynchronize(h->evDevUp)); CK(cudaStreamWaitEvent(st, h->evDevDone, 0)); h->devBusy = false; }
  return CUCD_OK;
}
int cucd_dev_me_sad_surface(cucd_handle* h, void* stream, int nPU, const cucd_me_desc* desc, uint32_t* d_sad) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !d_sad))) return fail(h, CUCD_ERR_INVALID, "cucd_dev_me_sad_surface: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  if (!h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_dev_me_sad_surface: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (dev_records_begin(h, st) != CUCD_OK) return CUCD_ERR_CUDA;
  size_t jobBytes, tileBytes; long long total, nTilesDy, nTilesO;
  const int rc = me_build_jobs(h, nPU, desc, h->hDevScratch, jobBytes, tileBytes, total, nTilesDy, nTilesO);
  if (rc != CUCD_OK) return rc;
  if (sync_ref_table(h) != CUCD_OK) return CUCD_ERR_CUDA;
  CK(h->dDevStage.reserve(jobBytes + 2 * tileBytes));
  CK(cudaMemcpyAsync(h->dDevStage.p, h->hDevScratch.p, jobBytes + 2 * tileBytes, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(h->evDevUp, st));
  MePlanes mp;
  mp.cur = h->dCur.p; mp.curStride = h->curStride; mp.ref = h->dRefPtr.p; mp.refStride = h->dRefStride.p; mp.bitDepth = h->cfg.bit_depth;
  const uint8_t* dAll = h->dDevStage.p;
  CK(launch_me_sad(mp, reinterpret_cast<const MeJob*>(dAll), nPU, reinterpret_cast<const int32_t*>(dAll + jobBytes), reinterpret_cast<const int32_t*>(dAll + jobBytes + tileBytes),
                   (int)nTilesDy, (int)nTilesO, d_sad, st, &h->launches));
  CK(cudaEventRecord(h->evDevDone, st)); h->devBusy = true;
  flush_launches(h);
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// Fractional-pel refinement: distortion of the 49 quarter-pel positions around an integer MV
// ------------------------------------------------------------------------------------------------
static int subpel_build_jobs(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, PinBuf<uint8_t>& scratch, bool ownBlocks = false, size_t* srcSamples = nullptr) {
  size_t blockOff = 0;
  const int W = h->cfg.width, H = h->cfg.height;
  CK(scratch.reserve((size_t)nPU * sizeof(SubpelJob) + 64));
  SubpelJob* jobs = reinterpret_cast<SubpelJob*>(scratch.p);
  for (int i = 0; i < nPU; i++) {
    const cucd_subpel_desc& d = desc[i];
    if (d.w < 4 || d.h < 4 || d.w > 64 || d.h > 64 || (d.w & 3) || (d.h & 3) || d.x < 0 || d.y < 0 || d.x + d.w > W || d.y + d.h > H)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost: bad PU");
    if (d.ref_idx < 0 || d.ref_idx >= (int)h->refs.size() || !h->refs[d.ref_idx].set) return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost: reference picture not set");
    const RefPlane& r = h->refs[d.ref_idx];
    if (d.x + d.mvx - 4 < -r.marginX || d.y + d.mvy - 4 < -r.marginY || d.x + d.mvx + d.w + 4 > W - 1 + r.marginX || d.y + d.mvy + d.h + 4 > H - 1 + r.marginY)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost: the interpolation support leaves the padded reference picture");
    SubpelJob& j = jobs[i];
    j.curOff = ownBlocks ? (int32_t)blockOff : d.y * h->curStride + d.x;
    blockOff += (size_t)d.w * d.h;
    j.refOff = (d.y + d.mvy + r.marginY) * r.stride + d.x + d.mvx + r.marginX;
    j.refSlot = d.ref_idx; j.w = (int16_t)d.w; j.h = (int16_t)d.h; j.useHadamard = d.use_hadamard ? 1 : 0;
  }
  if (blockOff > 0x7fffffffull) return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost_src: batch too large");
  if (srcSamples) *srcSamples = blockOff;
  return CUCD_OK;
}

static int me_subpel_cost_impl(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, const int16_t* src, uint32_t* cost) {
  const bool own = src != nullptr;
  if (!own && !h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  size_t srcSamples = 0;
  const int rc = subpel_build_jobs(h, nPU, desc, h->hScratch, own, &srcSamples);
  if (rc != CUCD_OK) return rc;
  if (sync_ref_table(h) != CUCD_OK) return CUCD_ERR_CUDA;
  BatchIo io(h);
  const int iJobs = io.add_in(h->hScratch.p, (size_t)nPU * sizeof(SubpelJob), true);
  const int iSrc = own ? io.add_in(src, srcSamples * sizeof(int16_t)) : -1;
  const int oCost = io.add_out(cost, (size_t)nPU * CUCD_SUBPEL_POINTS * sizeof(uint32_t));
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  MePlanes mp;
  mp.cur = own ? io.din<int16_t>(iSrc) : h->dCur.p; mp.curStride = own ? 0 : h->curStride;
  mp.ref = h->dRefPtr.p; mp.refStride = h->dRefStride.p; mp.bitDepth = h->cfg.bit_depth;
  if (!io.direct) CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_me_subpel(mp, io.din<SubpelJob>(iJobs), nPU, io.dout<uint32_t>(oCost), h->sMain, &h->launches));
  if (!io.direct) { CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true; } else h->kTimed = false;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}
int cucd_me_subpel_cost(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, uint32_t* cost) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !cost))) return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  return me_subpel_cost_impl(h, nPU, desc, nullptr, cost);
}
int cucd_me_subpel_cost_src(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, const int16_t* src, uint32_t* cost) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !src || !cost))) return fail(h, CUCD_ERR_INVALID, "cucd_me_subpel_cost_src: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  return me_subpel_cost_impl(h, nPU, desc, src, cost);
}

int cucd_dev_me_subpel_cost(cucd_handle* h, void* stream, int nPU, const cucd_subpel_desc* desc, uint32_t* d_cost) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !d_cost))) return fail(h, CUCD_ERR_INVALID, "cucd_dev_me_subpel_cost: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  if (!h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_dev_me_subpel_cost: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t st = (cudaStream_t)stream;
  if (dev_records_begin(h, st) != CUCD_OK) return CUCD_ERR_CUDA;
  const int rc = subpel_build_jobs(h, nPU, desc, h->hDevScratch);
  if (rc != CUCD_OK) return rc;
  if (sync_ref_table(h) != CUCD_OK) return CUCD_ERR_CUDA;
  const size_t bytes = (size_t)nPU * sizeof(SubpelJob);
  CK(h->dDevStage.reserve(bytes));
  CK(cudaMemcpyAsync(h->dDevStage.p, h->hDevScratch.p, bytes, cudaMemcpyHostToDevice, st));
  CK(cudaEventRecord(h->evDevUp, st));
  MePlanes mp;
  mp.cur = h->dCur.p; mp.curStride = h->curStride; mp.ref = h->dRefPtr.p; mp.refStride = h->dRefStride.p; mp.bitDepth = h->cfg.bit_depth;
  CK(launch_me_subpel(mp, reinterpret_cast<const SubpelJob*>(h->dDevStage.p), nPU, d_cost, st, &h->launches));
  CK(cudaEventRecord(h->evDevDone, st)); h->devBusy = true;
  flush_launches(h);
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// Motion compensation and distortion of inter candidates (uni- and bi-predictive), me_core.cuh me_mc_*
// ------------------------------------------------------------------------------------------------
int cucd_me_mc_cost(cucd_handle* h, int nPU, const cucd_mc_desc* desc, uint32_t* dist, int16_t* pred) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !dist))) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  if (!h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  const int W = h->cfg.width, H = h->cfg.height;
  // pinned scratch: [sorted jobs | CTA starts]; the jobs in caller order are built in a host vector first
  std::vector<McJob> jobs(nPU);
  long long predOff = 0;
  for (int i = 0; i < nPU; i++) {
    const cucd_mc_desc& d = desc[i];
    if (d.w < 4 || d.h < 4 || d.w > 64 || d.h > 64 || (d.w & 3) || (d.h & 3) || d.x < 0 || d.y < 0 || d.x + d.w > W || d.y + d.h > H)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: bad PU (w, h multiples of 4 in 4..64, inside the picture)");
    int nl = 0, slot[2], mvx[2], mvy[2], stride[2], mX[2], mY[2];
    for (int l = 0; l < 2; l++) {
      if (d.ref_idx[l] < 0) continue;
      if (d.ref_idx[l] >= (int)h->refs.size() || !h->refs[d.ref_idx[l]].set) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: reference picture not set");
      const RefPlane& r = h->refs[d.ref_idx[l]];
      const int ix = d.x + (d.mvx[l] >> 2), iy = d.y + (d.mvy[l] >> 2);
      if (ix - 3 < -r.marginX || iy - 3 < -r.marginY || ix + d.w + 3 > W - 1 + r.marginX || iy + d.h + 3 > H - 1 + r.marginY)
        return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: the interpolation support leaves the padded reference picture");
      slot[nl] = d.ref_idx[l]; mvx[nl] = d.mvx[l]; mvy[nl] = d.mvy[l]; stride[nl] = r.stride; mX[nl] = r.marginX; mY[nl] = r.marginY; nl++;
    }
    if (nl == 0) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_cost: a candidate uses neither list (ref_idx both < 0)");
    jobs[i] = me_mc_job(d.y * h->curStride + d.x, d.x, d.y, d.w, d.h, nl, slot, mvx, mvy, stride, mX, mY, d.use_hadamard, i, predOff);
    predOff += (long long)d.w * d.h;
  }
  const size_t jobBytes = up16((size_t)nPU * sizeof(McJob)), ctaBytes = up16((size_t)(nPU + 1) * sizeof(int32_t));
  CK(h->hScratch.reserve(jobBytes + ctaBytes));
  McJob* sorted = reinterpret_cast<McJob*>(h->hScratch.p);
  int32_t* ctaFirst = reinterpret_cast<int32_t*>(h->hScratch.p + jobBytes);
  const int nCta = me_mc_plan(nPU, jobs.data(), sorted, ctaFirst);
  if (sync_ref_table(h) != CUCD_OK) return CUCD_ERR_CUDA;
  BatchIo io(h);
  const int iAll = io.add_in(h->hScratch.p, jobBytes + ctaBytes, true);
  const int oDist = io.add_out(dist, (size_t)nPU * sizeof(uint32_t));
  const int oPred = io.add_out(pred, (size_t)predOff * sizeof(int16_t));
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  MePlanes mp;
  mp.cur = h->dCur.p; mp.curStride = h->curStride; mp.ref = h->dRefPtr.p; mp.refStride = h->dRefStride.p; mp.bitDepth = h->cfg.bit_depth;
  const uint8_t* dAll = io.din<uint8_t>(iAll);
  if (!io.direct) CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_me_mc(mp, reinterpret_cast<const McJob*>(dAll), reinterpret_cast<const int32_t*>(dAll + jobBytes), nCta, io.dout<uint32_t>(oDist),
                  pred ? io.dout<int16_t>(oPred) : nullptr, h->sMain, &h->launches));
  if (!io.direct) { CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true; } else h->kTimed = false;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// 4:2:0 chroma motion compensation and SSE of inter candidates, me_core.cuh me_mcc_*
// ------------------------------------------------------------------------------------------------
// one (W / 2) x (H / 2) plane whose first padded sample is `first` (stride in samples) into dst (pitch samples), pw x ph samples
static int upload_chroma_plane(cucd_handle* h, int16_t* dst, int pitch, const int16_t* first, int stride, int pw, int ph) {
  if (h->cfg.auto_pin_host) pin_host_range(h, first, ((size_t)(ph - 1) * stride + pw) * 2);
  CK(cudaMemcpy2DAsync(dst, (size_t)pitch * 2, first, (size_t)stride * 2, (size_t)pw * 2, ph, cudaMemcpyHostToDevice, h->sMain));
  return CUCD_OK;
}

int cucd_set_ref_picture_chroma(cucd_handle* h, int ref_idx, const int16_t* recCb, const int16_t* recCr, int strideC, int marginX, int marginY) {
  if (!h || ref_idx < 0 || ref_idx >= 64 || !recCb || !recCr || marginX < 0 || marginY < 0 || strideC < (h->cfg.width >> 1) + 2 * marginX)
    return fail(h, CUCD_ERR_INVALID, "cucd_set_ref_picture_chroma: bad argument");
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  if ((int)h->refCb.size() <= ref_idx) { h->refCb.resize(ref_idx + 1); h->refCr.resize(ref_idx + 1); }
  RefPlane* r[2] = {&h->refCb[ref_idx], &h->refCr[ref_idx]};
  const int16_t* src[2] = {recCb, recCr};
  const int pw = (h->cfg.width >> 1) + 2 * marginX, ph = (h->cfg.height >> 1) + 2 * marginY;
  const int pitch = (pw + 7) & ~7;
  r[0]->set = false;
  h->refTableCDirty = true;
  for (int c = 0; c < 2; c++) {
    CK(r[c]->buf.reserve((size_t)pitch * ph));
    if (upload_chroma_plane(h, r[c]->buf.p, pitch, src[c] - (ptrdiff_t)marginY * strideC - marginX, strideC, pw, ph) != CUCD_OK) return CUCD_ERR_CUDA;
  }
  CK(cudaStreamSynchronize(h->sMain));
  for (int c = 0; c < 2; c++) { r[c]->stride = pitch; r[c]->marginX = marginX; r[c]->marginY = marginY; r[c]->set = true; }
  return CUCD_OK;
}

int cucd_set_cur_picture_chroma(cucd_handle* h, const int16_t* orgCb, const int16_t* orgCr, int strideC) {
  if (!h || !orgCb || !orgCr || strideC < (h->cfg.width >> 1)) return fail(h, CUCD_ERR_INVALID, "cucd_set_cur_picture_chroma: bad argument");
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  const int wc = h->cfg.width >> 1, hc = h->cfg.height >> 1, pitch = (wc + 7) & ~7;
  h->curCSet = false;
  CK(h->dCurC.reserve((size_t)2 * pitch * hc));
  if (upload_chroma_plane(h, h->dCurC.p, pitch, orgCb, strideC, wc, hc) != CUCD_OK ||
      upload_chroma_plane(h, h->dCurC.p + (size_t)pitch * hc, pitch, orgCr, strideC, wc, hc) != CUCD_OK)
    return CUCD_ERR_CUDA;
  CK(cudaStreamSynchronize(h->sMain));
  h->curStrideC = pitch; h->curCSet = true;
  return CUCD_OK;
}

// the chroma twin of sync_ref_table: [2 slot + plane] plane pointers, [slot] strides
static int sync_ref_table_chroma(cucd_handle* h) {
  if (!h->refTableCDirty) return CUCD_OK;
  const size_t n = h->refCb.size();
  std::vector<const int16_t*> refPtr(2 * n, nullptr);
  std::vector<int32_t> refStride(n, 0);
  for (size_t i = 0; i < n; i++) { refPtr[2 * i] = h->refCb[i].buf.p; refPtr[2 * i + 1] = h->refCr[i].buf.p; refStride[i] = h->refCb[i].stride; }
  CK(h->dRefPtrC.reserve(std::max<size_t>(128, refPtr.size()))); CK(h->dRefStrideC.reserve(std::max<size_t>(64, refStride.size())));
  CK(cudaMemcpyAsync(h->dRefPtrC.p, refPtr.data(), refPtr.size() * sizeof(void*), cudaMemcpyHostToDevice, h->sMain));
  CK(cudaMemcpyAsync(h->dRefStrideC.p, refStride.data(), refStride.size() * 4, cudaMemcpyHostToDevice, h->sMain));
  CK(cudaStreamSynchronize(h->sMain));                 // the vectors above are about to go away
  h->refTableCDirty = false;
  return CUCD_OK;
}

int cucd_me_mc_chroma(cucd_handle* h, int nPU, const cucd_mc_desc* desc, uint32_t* sse, int16_t* pred) {
  if (!h || nPU < 0 || (nPU > 0 && (!desc || !sse))) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: bad argument");
  if (nPU == 0) return CUCD_OK;
  LOCK(h);
  if (!h->curCSet) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: cucd_set_cur_picture_chroma not called since the last cucd_set_cur_picture");
  CK(cudaSetDevice(h->cfg.device));
  const int W = h->cfg.width, H = h->cfg.height, Wc = W >> 1, Hc = H >> 1;
  std::vector<McJob> jobs(nPU);
  long long predOff = 0;
  for (int i = 0; i < nPU; i++) {
    const cucd_mc_desc& d = desc[i];
    if (d.w < 4 || d.h < 4 || d.w > 64 || d.h > 64 || (d.w & 3) || (d.h & 3) || d.x < 0 || d.y < 0 || d.x + d.w > W || d.y + d.h > H)
      return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: bad PU (w, h multiples of 4 in 4..64, inside the picture)");
    const int cx = d.x >> 1, cy = d.y >> 1, cw = d.w >> 1, ch = d.h >> 1;
    int nl = 0, slot[2], mvx[2], mvy[2], stride[2], mX[2], mY[2];
    for (int l = 0; l < 2; l++) {
      if (d.ref_idx[l] < 0) continue;
      if (d.ref_idx[l] >= (int)h->refCb.size() || !h->refCb[d.ref_idx[l]].set)
        return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: chroma of the reference picture not set (cucd_set_ref_picture_chroma after cucd_set_ref_picture)");
      const RefPlane& r = h->refCb[d.ref_idx[l]];
      const int ix = cx + (d.mvx[l] >> 3), iy = cy + (d.mvy[l] >> 3);
      if (ix - 1 < -r.marginX || iy - 1 < -r.marginY || ix + cw + 1 > Wc - 1 + r.marginX || iy + ch + 1 > Hc - 1 + r.marginY)
        return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: the interpolation support leaves the padded chroma plane");
      slot[nl] = d.ref_idx[l]; mvx[nl] = d.mvx[l]; mvy[nl] = d.mvy[l]; stride[nl] = r.stride; mX[nl] = r.marginX; mY[nl] = r.marginY; nl++;
    }
    if (nl == 0) return fail(h, CUCD_ERR_INVALID, "cucd_me_mc_chroma: a candidate uses neither list (ref_idx both < 0)");
    jobs[i] = me_mcc_job(cy * h->curStrideC + cx, cx, cy, cw, ch, nl, slot, mvx, mvy, stride, mX, mY, i, predOff);
    predOff += 2LL * cw * ch;
  }
  const size_t jobBytes = up16((size_t)nPU * sizeof(McJob)), ctaBytes = up16((size_t)(nPU + 1) * sizeof(int32_t));
  CK(h->hScratch.reserve(jobBytes + ctaBytes));
  McJob* sorted = reinterpret_cast<McJob*>(h->hScratch.p);
  int32_t* ctaFirst = reinterpret_cast<int32_t*>(h->hScratch.p + jobBytes);
  const int nCta = me_mcc_plan(nPU, jobs.data(), sorted, ctaFirst);
  if (sync_ref_table_chroma(h) != CUCD_OK) return CUCD_ERR_CUDA;
  BatchIo io(h);
  const int iAll = io.add_in(h->hScratch.p, jobBytes + ctaBytes, true);
  const int oSse = io.add_out(sse, (size_t)nPU * 2 * sizeof(uint32_t));
  const int oPred = io.add_out(pred, (size_t)predOff * sizeof(int16_t));
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  McChromaPlanes cp;
  cp.cur[0] = h->dCurC.p; cp.cur[1] = h->dCurC.p + (size_t)h->curStrideC * Hc; cp.curStride = h->curStrideC;
  cp.ref = h->dRefPtrC.p; cp.refStride = h->dRefStrideC.p; cp.bitDepth = h->cfg.bit_depth;
  const uint8_t* dAll = io.din<uint8_t>(iAll);
  if (!io.direct) CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_me_mc_chroma(cp, reinterpret_cast<const McJob*>(dAll), reinterpret_cast<const int32_t*>(dAll + jobBytes), nCta, io.dout<uint32_t>(oSse),
                         pred ? io.dout<int16_t>(oPred) : nullptr, h->sMain, &h->launches));
  if (!io.direct) { CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true; } else h->kTimed = false;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}

// ------------------------------------------------------------------------------------------------
// TU coding: intra TUs (xIntraCodingTUBlock) and the TUs of inter residual quadtrees (xEstimateResidualQT): forward half,
// reconstruction half, or the whole chain with the plain quantiser.  Inter calls (`inter`) pass the residual blocks as `org`,
// no border, and may ask for the SSE of the residual alone (`distZero`).
// ------------------------------------------------------------------------------------------------
static int tu_batch(cucd_handle* h, const char* who, int stage, int flags, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border,
                    int32_t* coefOut, const int32_t* levelIn, int16_t* pixOut, uint32_t* dist, int32_t* absSum, bool inter = false,
                    uint32_t* distZero = nullptr) {
  if (!h || nTU < 0 || (nTU > 0 && (!desc || !org || (!inter && !border)))) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": bad argument");
  if (nTU == 0) return CUCD_OK;
  if (inter && (flags & ~CUCD_TU_SIGN_HIDING))
    return fail(h, CUCD_ERR_INVALID, std::string(who) + ": flags may only hold CUCD_TU_SIGN_HIDING (an inter CU never lies in an I slice)");
  LOCK(h);
  CK(cudaSetDevice(h->cfg.device));
  // pass 1: validate, count per size class
  int count[6] = {0}, first[6] = {0};
  for (int i = 0; i < nTU; i++) {
    const cucd_tu_desc& d = desc[i];
    if (d.log2_size < 2 || d.log2_size > 5) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": log2_size must be 2..5");
    if (d.mode > 34 || d.qp < 0 || d.qp > 51) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": mode must be 0..34 and qp 0..51");
    if (inter && d.mode != 0) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": mode must be 0 (inter blocks are not predicted here)");
    if (inter && (d.flags & ~(CUCD_TU_TRANSFORM_SKIP | CUCD_TU_CHROMA))) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": unknown descriptor flags");
    if ((d.flags & CUCD_TU_TRANSFORM_SKIP) && d.log2_size != 2) return fail(h, CUCD_ERR_UNSUPPORTED, std::string(who) + ": transform skip is a 4x4 tool (log2MaxTransformSkipSize = 2)");
    count[d.log2_size]++;
  }
  for (int l = 3; l <= 5; l++) first[l] = first[l - 1] + count[l - 1];
  // pass 2: job records in size-class order straight into pinned scratch
  CK(h->hScratch.reserve((size_t)nTU * sizeof(TuJob) + 64));
  TuJob* jobs = reinterpret_cast<TuJob*>(h->hScratch.p);
  size_t orgOff = 0, borderOff = 0;
  {
    int next[6];
    for (int l = 2; l <= 5; l++) next[l] = first[l];
    for (int i = 0; i < nTU; i++) {
      const cucd_tu_desc& d = desc[i];
      TuJob& j = jobs[next[d.log2_size]++];
      j.orgOff = (int32_t)orgOff; j.borderOff = (int32_t)borderOff; j.outIndex = i; j.mode = d.mode; j.ts = d.flags & (CUCD_TU_TRANSFORM_SKIP | CUCD_TU_CHROMA); j.qp = d.qp; j.pad = 0;
      orgOff += (size_t)1 << (2 * d.log2_size); borderOff += ((size_t)4 << d.log2_size) + 1;
      if (orgOff > 0x7fff0000ull) return fail(h, CUCD_ERR_INVALID, std::string(who) + ": batch too large");
    }
  }
  BatchIo io(h);
  const int iOrg = io.add_in(org, orgOff * 2);
  const int iBrd = inter ? -1 : io.add_in(border, borderOff * 2);
  const int iJobs = io.add_in(jobs, (size_t)nTU * sizeof(TuJob), true);
  const int iLev = stage == 2 ? io.add_in(levelIn, orgOff * sizeof(int32_t)) : -1;
  io.inBytes += 256;
  // coefficient block: transform output (stage 0) / levels out (stage 1); stage 2 reads the uploaded levels in place
  const int oCoef = stage == 2 ? -1 : (coefOut ? io.add_out(coefOut, orgOff * sizeof(int32_t)) : io.add_scratch_out(orgOff * sizeof(int32_t)));
  const int oPix = (pixOut || stage != 0) ? (pixOut ? io.add_out(pixOut, orgOff * sizeof(int16_t)) : io.add_scratch_out(orgOff * sizeof(int16_t))) : -1;
  const int oDist = dist ? io.add_out(dist, (size_t)nTU * sizeof(uint32_t)) : io.add_scratch_out((size_t)nTU * sizeof(uint32_t));
  const int oAbs = absSum ? io.add_out(absSum, (size_t)nTU * sizeof(int32_t)) : io.add_scratch_out((size_t)nTU * sizeof(int32_t));
  const int oZero = distZero ? io.add_out(distZero, (size_t)nTU * sizeof(uint32_t)) : -1;
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  CK(cudaEventRecord(h->evK0, h->sMain));
  for (int l = 5; l >= 2; l--) {
    if (!count[l]) continue;
    TuBatch tb;
    tb.org = io.din<int16_t>(iOrg); tb.border = inter ? nullptr : io.din<int16_t>(iBrd); tb.jobs = io.din<TuJob>(iJobs) + first[l]; tb.count = count[l];
    tb.inter = inter ? 1 : 0; tb.distZero = oZero >= 0 ? io.dout<uint32_t>(oZero) : nullptr;
    tb.stage = stage; tb.bitDepth = h->cfg.bit_depth; tb.strong = h->cfg.strong_intra_smoothing;
    tb.intraSlice = (flags & CUCD_TU_INTRA_SLICE) ? 1 : 0; tb.signHiding = (flags & CUCD_TU_SIGN_HIDING) ? 1 : 0;
    tb.coef = stage == 2 ? io.din<int32_t>(iLev) : io.dout<int32_t>(oCoef);
    tb.pred = (stage == 0 && pixOut) ? io.dout<int16_t>(oPix) : nullptr;
    tb.reco = oPix >= 0 ? io.dout<int16_t>(oPix) : nullptr;
    tb.dist = io.dout<uint32_t>(oDist); tb.absSum = io.dout<int32_t>(oAbs);
    CK(launch_tu(l, tb, h->sMain, &h->launches));
  }
  CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}

int cucd_intra_tu_forward(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border, int32_t* coef, int16_t* pred) {
  if (nTU > 0 && !coef) return fail(h, CUCD_ERR_INVALID, "cucd_intra_tu_forward: coef is NULL");
  return tu_batch(h, "cucd_intra_tu_forward", 0, 0, nTU, desc, org, border, coef, nullptr, pred, nullptr, nullptr);
}
int cucd_intra_tu_recon(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border, const int32_t* level,
                        int16_t* reco, uint32_t* dist) {
  if (nTU > 0 && (!level || !reco || !dist)) return fail(h, CUCD_ERR_INVALID, "cucd_intra_tu_recon: NULL level / reco / dist");
  return tu_batch(h, "cucd_intra_tu_recon", 2, 0, nTU, desc, org, border, nullptr, level, reco, dist, nullptr);
}
int cucd_intra_tu_code(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border, int flags,
                       int32_t* level, int16_t* reco, uint32_t* dist, int32_t* abs_sum) {
  if (nTU > 0 && (!level || !reco || !dist)) return fail(h, CUCD_ERR_INVALID, "cucd_intra_tu_code: NULL level / reco / dist");
  return tu_batch(h, "cucd_intra_tu_code", 1, flags, nTU, desc, org, border, level, nullptr, reco, dist, abs_sum);
}
int cucd_inter_tu_forward(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi, int32_t* coef, uint32_t* dist_zero) {
  if (nTU > 0 && !coef) return fail(h, CUCD_ERR_INVALID, "cucd_inter_tu_forward: coef is NULL");
  return tu_batch(h, "cucd_inter_tu_forward", 0, 0, nTU, desc, resi, nullptr, coef, nullptr, nullptr, nullptr, nullptr, true, dist_zero);
}
int cucd_inter_tu_recon(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi, const int32_t* level, int16_t* rresi, uint32_t* dist) {
  if (nTU > 0 && (!level || !dist)) return fail(h, CUCD_ERR_INVALID, "cucd_inter_tu_recon: NULL level / dist");
  return tu_batch(h, "cucd_inter_tu_recon", 2, 0, nTU, desc, resi, nullptr, nullptr, level, rresi, dist, nullptr, true, nullptr);
}
int cucd_inter_tu_code(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi, int flags, int32_t* level, int16_t* rresi,
                       uint32_t* dist, uint32_t* dist_zero, int32_t* abs_sum) {
  if (nTU > 0 && (!level || !rresi || !dist)) return fail(h, CUCD_ERR_INVALID, "cucd_inter_tu_code: NULL level / rresi / dist");
  return tu_batch(h, "cucd_inter_tu_code", 1, flags, nTU, desc, resi, nullptr, level, nullptr, rresi, dist, abs_sum, true, dist_zero);
}

// ------------------------------------------------------------------------------------------------
// CU texture features (getTMVFeature) and AQ activity (TEncPreanalyzer) of the current picture
// ------------------------------------------------------------------------------------------------
int cucd_tmv_features(cucd_handle* h, int nCU, const cucd_cu_desc* cus, double* feat) {
  if (!h || nCU < 0 || (nCU > 0 && (!cus || !feat))) return fail(h, CUCD_ERR_INVALID, "cucd_tmv_features: bad argument");
  if (nCU == 0) return CUCD_OK;
  LOCK(h);
  if (!h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_tmv_features: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  CK(h->hScratch.reserve((size_t)nCU * sizeof(TmvCu) + 64));
  TmvCu* v = reinterpret_cast<TmvCu*>(h->hScratch.p);
  for (int i = 0; i < nCU; i++) {
    const cucd_cu_desc& c = cus[i];
    if (c.log2_size < 3 || c.log2_size > 6) return fail(h, CUCD_ERR_INVALID, "cucd_tmv_features: log2_size must be 3..6");
    const int n = 1 << c.log2_size;
    if (c.x < 0 || c.y < 0 || (c.x & (n - 1)) || (c.y & (n - 1)) || c.x + n > h->cfg.width || c.y + n > h->cfg.height)
      return fail(h, CUCD_ERR_INVALID, "cucd_tmv_features: CU must be aligned to its size and lie inside the picture");
    v[i].x = c.x; v[i].y = c.y; v[i].log2n = c.log2_size; v[i].pad = 0;
  }
  BatchIo io(h);
  const int iCus = io.add_in(v, (size_t)nCU * sizeof(TmvCu), true);
  const int oFeat = io.add_out(feat, (size_t)nCU * CUCD_TMV_FEATURES * sizeof(double));
  if (io.reserve() != CUCD_OK || io.upload(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_tmv_features(h->dCur.p, h->curStride, io.din<TmvCu>(iCus), nCU, io.dout<double>(oFeat), h->sMain, &h->launches));
  CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true;
  if (io.download(h->sMain) != CUCD_OK) return CUCD_ERR_CUDA;
  flush_launches(h);
  return CUCD_OK;
}

int cucd_aq_activity(cucd_handle* h, int max_aq_depth, double* const* activity, double* avg_activity) {
  if (!h || max_aq_depth < 1 || max_aq_depth > 4 || (!activity && !avg_activity)) return fail(h, CUCD_ERR_INVALID, "cucd_aq_activity: bad argument");
  LOCK(h);
  if (!h->curSet) return fail(h, CUCD_ERR_INVALID, "cucd_aq_activity: cucd_set_cur_picture not called");
  CK(cudaSetDevice(h->cfg.device));
  const int W = h->cfg.width, H = h->cfg.height;
  AqLayers L; L.count = max_aq_depth; L.total = 0;
  for (int d = 0; d < 4; d++) { L.part[d] = 0; L.off[d] = 0; }
  for (int d = 0; d < max_aq_depth; d++) {
    L.part[d] = h->cfg.ctu_size >> d; L.off[d] = L.total;
    L.total += ((W + L.part[d] - 1) / L.part[d]) * ((H + L.part[d] - 1) / L.part[d]);
  }
  for (int d = max_aq_depth; d <= 4; d++) L.off[d] = L.total;
  CK(h->hScratch.reserve((size_t)L.total * sizeof(double) + 64));
  double* act = reinterpret_cast<double*>(h->hScratch.p);
  CK(h->bOut.reserve((size_t)L.total * 2 + 64));
  double* dAct = reinterpret_cast<double*>(h->bOut.p);
  CK(cudaEventRecord(h->evK0, h->sMain));
  CK(launch_aq_activity(h->dCur.p, h->curStride, W, H, L, dAct, h->sMain, &h->launches));
  CK(cudaEventRecord(h->evK1, h->sMain)); h->kTimed = true;
  CK(cudaMemcpyAsync(act, dAct, (size_t)L.total * sizeof(double), cudaMemcpyDeviceToHost, h->sMain));
  CK(cudaStreamSynchronize(h->sMain));
  for (int d = 0; d < max_aq_depth; d++) {
    const int n = L.off[d + 1] - L.off[d];
    if (activity && activity[d]) memcpy(activity[d], act + L.off[d], (size_t)n * sizeof(double));
    if (avg_activity) {          // dSumAct accumulates in raster order (TEncPreanalyzer.cpp:132): a sequential double sum, kept on the host
      double sum = 0.0;
      for (int i = 0; i < n; i++) sum += act[L.off[d] + i];
      avg_activity[d] = sum / (double)(unsigned)n;
    }
  }
  flush_launches(h);
  return CUCD_OK;
}

}  // extern "C"
