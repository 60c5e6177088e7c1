// server.cpp - cucd_server: the coalescing host runtime of libcucudecide.so (SURVEY.md 8f.1, include/cucd_ipc.h).
//
// One process owns the GPU.  N encoder instances (processes; HM is single-threaded and not re-entrant) map the shared-memory
// segment this program creates, post their requests and sleep.  The server loop polls the slots:
//   - S2 requests (rough mode decision of a few PUs with caller-supplied borders - what TEncSearch.cpp:2327-2361 can offer at a
//     time) of ALL instances are gathered for a short batching window and run as ONE cucd_intra_rmd_batch per bit depth;
//   - S1 / S3 / sub-pel / inter-candidate requests depend on their instance's pictures and run on that instance's handle, in arrival order.
// Only the C ABI of include/cucudecide.h is used: the server is an ordinary client of the library.
//
//   cucd_server --name /cucd_xyz --clients N [--window-us 20] [--device 0]      prints one JSON line of statistics on exit
#include <cuda_runtime.h>
#include <chrono>
#include <csignal>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>
#include "../../include/cucd_ipc.h"

namespace {

volatile sig_atomic_t g_stop = 0;
void on_signal(int) { g_stop = 1; }

struct Client {
  cucd_handle* h = nullptr;      // S1 / S3 / sub-pel state of this instance
  int W = 0, H = 0, bd = 0, strong = 0;
  bool open = false, closed = false;
};

struct PinnedVec {               // grow-only pinned host array
  unsigned char* p = nullptr; size_t cap = 0;
  unsigned char* reserve(size_t n) {
    if (n <= cap) return p;
    if (p) cudaFreeHost(p);
    cap = n * 2 + 4096;
    if (cudaMallocHost(&p, cap) != cudaSuccess) { p = nullptr; cap = 0; }
    return p;
  }
};

void reply(cucd_ipc_slot& s, int status, const char* err) {
  s.status = status;
  if (err) { strncpy(s.err, err, sizeof s.err - 1); s.err[sizeof s.err - 1] = 0; } else s.err[0] = 0;
  s.state.store(CUCD_IPC_DONE, std::memory_order_release);
  cucd_futex(&s.state, FUTEX_WAKE, INT_MAX);
}

double now_us() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

}  // namespace

int main(int argc, char** argv) {
  std::string name = "/cucd_server";
  int clients = 8, device = 0; double windowUs = 20.0;
  for (int i = 1; i + 1 < argc; i += 2) {
    if (!strcmp(argv[i], "--name")) name = argv[i + 1];
    else if (!strcmp(argv[i], "--clients")) clients = atoi(argv[i + 1]);
    else if (!strcmp(argv[i], "--window-us")) windowUs = atof(argv[i + 1]);
    else if (!strcmp(argv[i], "--device")) device = atoi(argv[i + 1]);
  }
  if (clients < 1 || clients > CUCD_IPC_MAX_CLIENTS) { fprintf(stderr, "cucd_server: --clients must be 1..%d\n", CUCD_IPC_MAX_CLIENTS); return 2; }
  signal(SIGTERM, on_signal); signal(SIGINT, on_signal);

  shm_unlink(name.c_str());
  const int fd = shm_open(name.c_str(), O_CREAT | O_EXCL | O_RDWR, 0600);
  if (fd < 0) { perror("cucd_server: shm_open"); return 2; }
  const size_t total = cucd_ipc_total_bytes(clients);
  if (ftruncate(fd, (off_t)total) != 0) { perror("cucd_server: ftruncate"); shm_unlink(name.c_str()); return 2; }
  void* mem = mmap(nullptr, total, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
  close(fd);
  if (mem == MAP_FAILED) { perror("cucd_server: mmap"); shm_unlink(name.c_str()); return 2; }
  cucd_ipc_header* hdr = new (mem) cucd_ipc_header;
  hdr->magic = CUCD_IPC_MAGIC; hdr->version = CUCD_IPC_VERSION; hdr->max_clients = (uint32_t)clients; hdr->arena_bytes = CUCD_IPC_ARENA_BYTES;
  hdr->next_client.store(0);
  for (int i = 0; i < CUCD_IPC_MAX_CLIENTS; i++) hdr->slot[i].state.store(CUCD_IPC_FREE);

  // the shared S2 handles (one per bit depth seen); created on the first OPEN so that a wrong device fails loudly there
  cucd_handle* rmdHandle[3] = {nullptr, nullptr, nullptr};      // bit depth 8, 9, 10
  std::vector<Client> cl(clients);
  if (cudaSetDevice(device) != cudaSuccess) { fprintf(stderr, "cucd_server: no CUDA device %d - the library has no CPU path\n", device); shm_unlink(name.c_str()); return 3; }
  // Page-lock the whole segment: requests and replies are then DMA'd straight from / to the instances' arenas
  const bool segPinned = cudaHostRegister(mem, total, cudaHostRegisterDefault) == cudaSuccess;
  if (!segPinned) cudaGetLastError();
  hdr->server_ready.store(1, std::memory_order_release);

  PinnedVec stDesc, stOrg, stBrd, stSad;
  long long nReq[16] = {0}, rmdBatches = 0, rmdPus = 0, rmdReqs = 0, maxBatchPus = 0;
  double rmdBusyUs = 0, t0 = now_us();
  int nClosed = 0, nSeen = 0;
  std::vector<int> pendingRmd;
  double firstRmdSeen = 0;

  while (!g_stop) {
    bool any = false;
    const int claimed = std::min<int>((int)hdr->next_client.load(std::memory_order_acquire), clients);
    nSeen = claimed;
    for (int c = 0; c < claimed; c++) {
      cucd_ipc_slot& s = hdr->slot[c];
      if (s.state.load(std::memory_order_acquire) != CUCD_IPC_READY) continue;
      Client& k = cl[c];
      unsigned char* in = cucd_ipc_arena(hdr, c);
      unsigned char* out = in + s.out_off;
      if (s.op == CUCD_IPC_RMD) {                                   // gathered below
        bool listed = false;
        for (int p : pendingRmd) listed = listed || p == c;
        if (!listed) { if (pendingRmd.empty()) firstRmdSeen = now_us(); pendingRmd.push_back(c); }
        continue;
      }
      any = true;
      nReq[s.op & 15]++;
      switch (s.op) {
        case CUCD_IPC_OPEN: {
          if (k.h && (k.W != s.args[0] || k.H != s.args[1] || k.bd != s.args[2] || k.strong != s.args[3])) { cucd_destroy(k.h); k.h = nullptr; }
          int rc = CUCD_OK;
          if (!k.h) {
            cucd_config cfg = {s.args[0], s.args[1], s.args[2], 64, 4, s.args[3], device, 1, 1, 0};
            rc = cucd_create(&cfg, &k.h);
            k.W = s.args[0]; k.H = s.args[1]; k.bd = s.args[2]; k.strong = s.args[3];
          }
          const int bi = k.bd - 8;
          if (rc == CUCD_OK && bi >= 0 && bi < 3 && !rmdHandle[bi]) {
            cucd_config cfg = {64, 64, k.bd, 64, 4, k.strong, device, 1, 1, 0};     // S2 batches carry their own samples: the picture size is irrelevant
            rc = cucd_create(&cfg, &rmdHandle[bi]);
          }
          k.open = rc == CUCD_OK;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(nullptr));
          break;
        }
        case CUCD_IPC_CLOSE:
          if (k.h) { cucd_destroy(k.h); k.h = nullptr; }
          k.closed = true; nClosed++;
          reply(s, CUCD_OK, nullptr);
          break;
        case CUCD_IPC_FRAME: {
          cucd_frame_out fo; memset(&fo, 0, sizeof fo);
          fo.obf = reinterpret_cast<int16_t*>(out);
          fo.outlier = reinterpret_cast<int16_t*>(out) + (size_t)(k.W / 4) * (k.H / 4);
          const int rc = k.h ? cuCUDecide_frame(k.h, reinterpret_cast<const int16_t*>(in), k.W, nullptr, 0, 0, &fo) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_SET_CUR: {
          const int rc = k.h ? cucd_set_cur_picture(k.h, reinterpret_cast<const int16_t*>(in), k.W) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_SET_REF: {
          const int mx = s.args[1], my = s.args[2], pw = k.W + 2 * mx;
          const int rc = k.h ? cucd_set_ref_picture(k.h, s.args[0], reinterpret_cast<const int16_t*>(in) + (size_t)my * pw + mx, pw, mx, my) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_ME_SURFACE: {
          const int rc = k.h ? cucd_me_sad_surface(k.h, s.n, reinterpret_cast<const cucd_me_desc*>(in), reinterpret_cast<uint32_t*>(out)) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_SUBPEL: {
          const int rc = k.h ? cucd_me_subpel_cost(k.h, s.n, reinterpret_cast<const cucd_subpel_desc*>(in), reinterpret_cast<uint32_t*>(out)) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_MC: {
          // the reply must fit what the client reserved: dist, then (args[0]) the predictions
          const size_t nC = (size_t)(s.n > 0 ? s.n : 0), distBytes = (nC * 4 + 15) & ~(size_t)15;
          const cucd_mc_desc* desc = reinterpret_cast<const cucd_mc_desc*>(in);
          size_t need = distBytes;
          if (nC * sizeof(cucd_mc_desc) <= s.in_bytes && s.args[0])
            for (size_t i = 0; i < nC; i++) need += (size_t)(desc[i].w > 0 ? desc[i].w : 0) * (size_t)(desc[i].h > 0 ? desc[i].h : 0) * 2;
          if (nC * sizeof(cucd_mc_desc) > s.in_bytes || need > s.out_bytes || s.out_off + s.out_bytes > hdr->arena_bytes) {
            reply(s, CUCD_ERR_INVALID, "cucd_me_mc_cost: request and reply sizes disagree");
            break;
          }
          int16_t* pred = s.args[0] ? reinterpret_cast<int16_t*>(out + distBytes) : nullptr;
          const int rc = k.h ? cucd_me_mc_cost(k.h, s.n, desc, reinterpret_cast<uint32_t*>(out), pred) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_SET_REF_CHROMA: {
          // margins come from the client: bound them by the arena and size the planes in 64 bits, so that a huge margin fails the
          // size check instead of overflowing
          const int mx = s.args[1], my = s.args[2];
          const long long pw64 = k.W / 2 + 2LL * mx, ph64 = k.H / 2 + 2LL * my;
          if (mx < 0 || my < 0 || (unsigned long long)mx > hdr->arena_bytes || (unsigned long long)my > hdr->arena_bytes ||
              s.in_bytes > hdr->arena_bytes || (unsigned long long)(pw64 * ph64) * 4 > s.in_bytes) {
            reply(s, CUCD_ERR_INVALID, "cucd_set_ref_picture_chroma: request size disagrees");
            break;
          }
          const int pw = (int)pw64, ph = (int)ph64;                  // both planes fit the arena: far below 2^31
          const int16_t* cb = reinterpret_cast<const int16_t*>(in) + (size_t)my * pw + mx;
          const int rc = k.h ? cucd_set_ref_picture_chroma(k.h, s.args[0], cb, cb + (size_t)pw * ph, pw, mx, my) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_SET_CUR_CHROMA: {
          const size_t plane = (size_t)(k.W / 2) * (k.H / 2);
          if (2 * plane * 2 > s.in_bytes) { reply(s, CUCD_ERR_INVALID, "cucd_set_cur_picture_chroma: request size disagrees"); break; }
          const int16_t* cb = reinterpret_cast<const int16_t*>(in);
          const int rc = k.h ? cucd_set_cur_picture_chroma(k.h, cb, cb + plane, k.W / 2) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        case CUCD_IPC_MC_CHROMA: {
          // the reply must fit what the client reserved: sse, then (args[0]) the Cb and Cr predictions
          const size_t nC = (size_t)(s.n > 0 ? s.n : 0), sseBytes = (nC * 8 + 15) & ~(size_t)15;
          const cucd_mc_desc* desc = reinterpret_cast<const cucd_mc_desc*>(in);
          size_t need = sseBytes;
          if (nC * sizeof(cucd_mc_desc) <= s.in_bytes && s.args[0])
            for (size_t i = 0; i < nC; i++) need += 2 * (size_t)(desc[i].w > 0 ? desc[i].w / 2 : 0) * (size_t)(desc[i].h > 0 ? desc[i].h / 2 : 0) * 2;
          if (nC * sizeof(cucd_mc_desc) > s.in_bytes || need > s.out_bytes || s.out_off + s.out_bytes > hdr->arena_bytes) {
            reply(s, CUCD_ERR_INVALID, "cucd_me_mc_chroma: request and reply sizes disagree");
            break;
          }
          int16_t* pred = s.args[0] ? reinterpret_cast<int16_t*>(out + sseBytes) : nullptr;
          const int rc = k.h ? cucd_me_mc_chroma(k.h, s.n, desc, reinterpret_cast<uint32_t*>(out), pred) : CUCD_ERR_INVALID;
          reply(s, rc, rc == CUCD_OK ? nullptr : cucd_last_error(k.h));
          break;
        }
        default:
          reply(s, CUCD_ERR_INVALID, "unknown request");
      }
    }
    // ---- S2: one batch for everything gathered.  The window closes when every open instance is waiting, or after windowUs.
    if (!pendingRmd.empty()) {
      int openNow = 0;
      for (int c = 0; c < claimed; c++) openNow += cl[c].open && !cl[c].closed;
      if ((int)pendingRmd.size() >= openNow || now_us() - firstRmdSeen >= windowUs) {
        const double tb = now_us();
        for (int bi = 0; bi < 3; bi++) {
          size_t nPu = 0, orgN = 0, brdN = 0;
          for (int c : pendingRmd) if (cl[c].bd - 8 == bi) { const cucd_ipc_slot& s = hdr->slot[c]; nPu += (size_t)s.n; orgN += (size_t)s.args[0]; brdN += (size_t)s.args[1]; }
          if (!nPu) continue;
          cucd_pu_desc* desc = reinterpret_cast<cucd_pu_desc*>(stDesc.reserve(nPu * sizeof(cucd_pu_desc)));
          int16_t* org = reinterpret_cast<int16_t*>(stOrg.reserve(orgN * 2 + 64));
          int16_t* brd = reinterpret_cast<int16_t*>(stBrd.reserve(brdN * 2 + 64));
          uint32_t* sad = reinterpret_cast<uint32_t*>(stSad.reserve(nPu * 35 * 4));
          size_t pu = 0, oo = 0, bo = 0;
          int rc = (desc && org && brd && sad && rmdHandle[bi]) ? CUCD_OK : CUCD_ERR_NOMEM;
          if (rc == CUCD_OK) {
            for (int c : pendingRmd) if (cl[c].bd - 8 == bi) {
              const cucd_ipc_slot& s = hdr->slot[c];
              const unsigned char* in = cucd_ipc_arena(hdr, c);
              const size_t o0 = ((size_t)s.n * sizeof(cucd_pu_desc) + 15) & ~(size_t)15;
              memcpy(desc + pu, in, (size_t)s.n * sizeof(cucd_pu_desc));
              memcpy(org + oo, in + o0, (size_t)s.args[0] * 2);
              memcpy(brd + bo, in + o0 + (size_t)s.args[0] * 2, (size_t)s.args[1] * 2);
              pu += (size_t)s.n; oo += (size_t)s.args[0]; bo += (size_t)s.args[1];
            }
            rc = cucd_intra_rmd_batch(rmdHandle[bi], (int)nPu, desc, org, brd, sad);
          }
          pu = 0;
          for (int c : pendingRmd) if (cl[c].bd - 8 == bi) {
            cucd_ipc_slot& s = hdr->slot[c];
            if (rc == CUCD_OK) memcpy(cucd_ipc_arena(hdr, c) + s.out_off, sad + pu * 35, (size_t)s.n * 35 * 4);
            pu += (size_t)s.n;
            reply(s, rc, rc == CUCD_OK ? nullptr : (rmdHandle[bi] ? cucd_last_error(rmdHandle[bi]) : "no S2 handle"));
            rmdReqs++;
          }
          rmdBatches++; rmdPus += (long long)nPu; if ((long long)nPu > maxBatchPus) maxBatchPus = (long long)nPu;
        }
        rmdBusyUs += now_us() - tb;
        pendingRmd.clear();
        any = true;
      }
    }
    if (nSeen > 0 && nClosed >= nSeen && nClosed >= 1 && (int)hdr->next_client.load() <= nClosed) {
      // every instance that ever connected has closed; give late starters a moment, then leave
      static double idleSince = 0;
      if (!idleSince) idleSince = now_us();
      if (now_us() - idleSince > 2e6 || nClosed >= clients) break;
    }
    if (!any && pendingRmd.empty()) __builtin_ia32_pause();
  }
  long long launches = 0;
  for (auto& k : cl) if (k.h) { launches += cucd_launch_count(k.h); cucd_destroy(k.h); }
  for (auto* h : rmdHandle) if (h) { launches += cucd_launch_count(h); cucd_destroy(h); }
  if (segPinned) cudaHostUnregister(mem);
  printf("{\"clients\": %d, \"closed\": %d, \"seconds\": %.3f, \"rmd_requests\": %lld, \"rmd_pus\": %lld, \"rmd_batches\": %lld, \"pus_per_batch\": %.1f, "
         "\"requests_per_batch\": %.2f, \"max_batch_pus\": %lld, \"rmd_busy_seconds\": %.3f, \"frames\": %lld, \"me_surfaces\": %lld, \"subpel\": %lld, "
         "\"mc\": %lld, \"mc_chroma\": %lld, \"set_ref\": %lld, \"window_us\": %.1f, \"segment_pinned\": %s}\n",
         nSeen, nClosed, (now_us() - t0) * 1e-6, rmdReqs, rmdPus, rmdBatches, rmdBatches ? (double)rmdPus / rmdBatches : 0.0,
         rmdBatches ? (double)rmdReqs / rmdBatches : 0.0, maxBatchPus, rmdBusyUs * 1e-6, nReq[CUCD_IPC_FRAME], nReq[CUCD_IPC_ME_SURFACE], nReq[CUCD_IPC_SUBPEL],
         nReq[CUCD_IPC_MC], nReq[CUCD_IPC_MC_CHROMA], nReq[CUCD_IPC_SET_REF], windowUs, segPinned ? "true" : "false");
  munmap(mem, total);
  shm_unlink(name.c_str());
  return 0;
}
