/* cucd_ipc.h - shared-memory protocol between encoder instances and cucd_server, the coalescing host runtime of
 * libcucudecide.so (SURVEY.md 8f.1).
 *
 * Why: in the live encoder a PU's reference border is an intermediate state of the reconstruction, so ONE instance can only
 * offer the few PUs of its current CU at a time (TEncSearch.cpp:2327-2361 is entered once per PU).  HM is single-threaded and
 * not re-entrant (global state: g_bitDepth, g_iPOC, g_bDecisionSwitch ..., TComRom.cpp:253-260), so concurrency means several
 * encoder PROCESSES - one per picture / intra period in flight - and only one process should own the GPU context.  cucd_server
 * owns the device and the handles; every encoder instance maps the same POSIX shared-memory segment, posts its request into its
 * own slot + arena and sleeps on a futex; the server turns everything that is pending into one batch per request kind.
 *   S2  (cucd_intra_rmd_batch)   stateless: requests of ALL instances with the same bit depth are coalesced into one batch
 *   S1  (cuCUDecide_frame), S3 (cucd_set_cur/ref_picture, cucd_me_sad_surface), sub-pel (cucd_me_subpel_cost), inter candidates
 *        (cucd_me_mc_cost, cucd_set_ref/cur_picture_chroma, cucd_me_mc_chroma), motion search (cucd_me_search, cucd_me_tz_search; the _src form stays
 *        in process): served on the instance's own handle inside the server (they depend on that instance's pictures), in
 *        arrival order.  A server that predates an op answers it with CUCD_ERR_INVALID, "unknown request".
 * The client side below is header-only C++ (what the reference's shim includes); the entry points mirror the C ABI of
 * include/cucudecide.h one to one, so an integration switches between in-process and server mode without other changes.
 */
#ifndef CUCD_IPC_H
#define CUCD_IPC_H
#include <atomic>
#include <cerrno>
#include <climits>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <linux/futex.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <unistd.h>
#include "cucudecide.h"

#define CUCD_IPC_MAGIC 0x43554344u
#define CUCD_IPC_VERSION 1u
#define CUCD_IPC_MAX_CLIENTS 64
#define CUCD_IPC_ARENA_BYTES ((size_t)96 << 20)      /* request + reply payload of one instance (a padded 2160p plane is 34 MB) */

enum cucd_ipc_op { CUCD_IPC_OPEN = 1, CUCD_IPC_CLOSE, CUCD_IPC_FRAME, CUCD_IPC_RMD, CUCD_IPC_SET_CUR, CUCD_IPC_SET_REF, CUCD_IPC_ME_SURFACE, CUCD_IPC_SUBPEL,
                   CUCD_IPC_MC, CUCD_IPC_SET_REF_CHROMA, CUCD_IPC_SET_CUR_CHROMA, CUCD_IPC_MC_CHROMA, CUCD_IPC_ME_SEARCH,
                   CUCD_IPC_ME_TZ_SEARCH };
enum cucd_ipc_state { CUCD_IPC_FREE = 0, CUCD_IPC_IDLE = 1, CUCD_IPC_READY = 2, CUCD_IPC_DONE = 3, CUCD_IPC_CLOSED = 4 };

struct alignas(128) cucd_ipc_slot {
  std::atomic<uint32_t> state;   /* cucd_ipc_state; the futex word */
  uint32_t op;                   /* cucd_ipc_op */
  int32_t status;                /* cucd_status of the reply */
  int32_t n;                     /* PUs / pictures of the request */
  int32_t args[12];              /* op-specific scalars */
  uint64_t in_bytes, out_bytes;  /* payload sizes inside the arena: request at offset 0, reply at offset out_off */
  uint64_t out_off;
  char err[160];
};
struct cucd_ipc_header {
  uint32_t magic, version, max_clients, pad;
  std::atomic<uint32_t> server_ready, next_client;
  uint64_t arena_bytes;
  cucd_ipc_slot slot[CUCD_IPC_MAX_CLIENTS];
};
static inline size_t cucd_ipc_total_bytes(int clients) { return sizeof(cucd_ipc_header) + (size_t)clients * CUCD_IPC_ARENA_BYTES; }
static inline unsigned char* cucd_ipc_arena(cucd_ipc_header* h, int client) {
  return reinterpret_cast<unsigned char*>(h) + sizeof(cucd_ipc_header) + (size_t)client * h->arena_bytes;
}
static inline long cucd_futex(std::atomic<uint32_t>* addr, int op, uint32_t val) {
  return syscall(SYS_futex, reinterpret_cast<uint32_t*>(addr), op, val, (void*)0, (void*)0, 0);
}

/* ---- client ------------------------------------------------------------------------------------------------------------- */
struct cucd_ipc_client {
  cucd_ipc_header* hdr; int id; cucd_ipc_slot* s; unsigned char* arena; char err[160];
  cucd_ipc_client() : hdr(0), id(-1), s(0), arena(0) { err[0] = 0; }
  bool connected() const { return hdr != 0; }

  /* attach to the segment named by `name` (shm_open name, e.g. "/cucd_1234") and claim a slot */
  int connect(const char* name) {
    const int fd = shm_open(name, O_RDWR, 0600);
    if (fd < 0) { snprintf(err, sizeof err, "shm_open(%s): %s", name, strerror(errno)); return CUCD_ERR_INVALID; }
    struct stat st;
    if (fstat(fd, &st) != 0 || (size_t)st.st_size < sizeof(cucd_ipc_header)) { close(fd); snprintf(err, sizeof err, "bad segment"); return CUCD_ERR_INVALID; }
    void* p = mmap(0, (size_t)st.st_size, PROT_READ | PROT_WRITE, MAP_SHARED, fd, 0);
    close(fd);
    if (p == MAP_FAILED) { snprintf(err, sizeof err, "mmap: %s", strerror(errno)); return CUCD_ERR_NOMEM; }
    hdr = static_cast<cucd_ipc_header*>(p);
    if (hdr->magic != CUCD_IPC_MAGIC || hdr->version != CUCD_IPC_VERSION) { snprintf(err, sizeof err, "protocol mismatch"); hdr = 0; return CUCD_ERR_INVALID; }
    for (int spin = 0; !hdr->server_ready.load(std::memory_order_acquire); spin++) { if (spin > 100000) { snprintf(err, sizeof err, "server not ready"); hdr = 0; return CUCD_ERR_INVALID; } usleep(100); }
    id = (int)hdr->next_client.fetch_add(1);
    if (id >= (int)hdr->max_clients) { snprintf(err, sizeof err, "no free client slot"); hdr = 0; return CUCD_ERR_INVALID; }
    s = &hdr->slot[id]; arena = cucd_ipc_arena(hdr, id);
    s->state.store(CUCD_IPC_IDLE, std::memory_order_release);
    return CUCD_OK;
  }
  /* post the request that has been written into the slot / arena and sleep until the reply is there */
  int call(uint32_t op, int n, uint64_t in_bytes, uint64_t out_bytes) {
    s->op = op; s->n = n; s->in_bytes = in_bytes; s->out_bytes = out_bytes; s->out_off = (in_bytes + 255) & ~(uint64_t)255;
    if (s->out_off + out_bytes > hdr->arena_bytes) { snprintf(err, sizeof err, "request of %llu + %llu bytes exceeds the arena", (unsigned long long)in_bytes, (unsigned long long)out_bytes); return CUCD_ERR_NOMEM; }
    s->state.store(CUCD_IPC_READY, std::memory_order_release);
    for (int spin = 0;; spin++) {
      const uint32_t v = s->state.load(std::memory_order_acquire);
      if (v == CUCD_IPC_DONE) break;
      if (spin < 4000) { __builtin_ia32_pause(); continue; }
      cucd_futex(&s->state, FUTEX_WAIT, v);          /* returns at once if the state moved on meanwhile */
    }
    s->state.store(CUCD_IPC_IDLE, std::memory_order_relaxed);
    if (s->status != CUCD_OK) { memcpy(err, s->err, sizeof err); err[sizeof err - 1] = 0; }
    return s->status;
  }
  const unsigned char* reply() const { return arena + s->out_off; }

  /* ---- the C ABI, one to one ---- */
  int open(int W, int H, int bitDepth, int strong) {
    s->args[0] = W; s->args[1] = H; s->args[2] = bitDepth; s->args[3] = strong;
    return call(CUCD_IPC_OPEN, 0, 0, 0);
  }
  void close_client() { if (hdr) { call(CUCD_IPC_CLOSE, 0, 0, 0); s->state.store(CUCD_IPC_CLOSED, std::memory_order_release); hdr = 0; } }
  /* cuCUDecide_frame(org, stride, no reconstruction): OBF (W/4 x H/4) and Outlier (W x H) planes back, tight */
  int frame(int W, int H, const int16_t* org, int stride, int16_t* obf, int16_t* outlier) {
    for (int r = 0; r < H; r++) memcpy(arena + (size_t)r * W * 2, org + (size_t)r * stride, (size_t)W * 2);
    const size_t nObf = (size_t)(W / 4) * (H / 4), nOut = (size_t)W * H;
    const int rc = call(CUCD_IPC_FRAME, 1, nOut * 2, (nObf + nOut) * 2);
    if (rc == CUCD_OK) { memcpy(obf, reply(), nObf * 2); memcpy(outlier, reply() + nObf * 2, nOut * 2); }
    return rc;
  }
  int intra_rmd_batch(int nPU, const cucd_pu_desc* desc, const int16_t* org, const int16_t* border, uint32_t* sad) {
    size_t orgN = 0, brdN = 0;
    for (int i = 0; i < nPU; i++) { orgN += (size_t)1 << (2 * desc[i].log2_size); brdN += ((size_t)4 << desc[i].log2_size) + 1; }
    unsigned char* p = arena;                         /* [desc | pad | org | border] */
    memcpy(p, desc, (size_t)nPU * sizeof(cucd_pu_desc));
    const size_t o0 = ((size_t)nPU * sizeof(cucd_pu_desc) + 15) & ~(size_t)15;
    memcpy(p + o0, org, orgN * 2); memcpy(p + o0 + orgN * 2, border, brdN * 2);
    s->args[0] = (int32_t)orgN; s->args[1] = (int32_t)brdN;
    const int rc = call(CUCD_IPC_RMD, nPU, o0 + (orgN + brdN) * 2, (size_t)nPU * 35 * 4);
    if (rc == CUCD_OK) memcpy(sad, reply(), (size_t)nPU * 35 * 4);
    return rc;
  }
  int set_cur_picture(int W, int H, const int16_t* org, int stride) {
    for (int r = 0; r < H; r++) memcpy(arena + (size_t)r * W * 2, org + (size_t)r * stride, (size_t)W * 2);
    return call(CUCD_IPC_SET_CUR, 1, (size_t)W * H * 2, 0);
  }
  int set_ref_picture(int W, int H, int ref_idx, const int16_t* recY, int stride, int marginX, int marginY) {
    const int pw = W + 2 * marginX, ph = H + 2 * marginY;
    const int16_t* first = recY - (ptrdiff_t)marginY * stride - marginX;
    for (int r = 0; r < ph; r++) memcpy(arena + (size_t)r * pw * 2, first + (size_t)r * stride, (size_t)pw * 2);
    s->args[0] = ref_idx; s->args[1] = marginX; s->args[2] = marginY;
    return call(CUCD_IPC_SET_REF, 1, (size_t)pw * ph * 2, 0);
  }
  int me_sad_surface(int nPU, const cucd_me_desc* desc, uint32_t* sadOut) {
    size_t total = 0;
    for (int i = 0; i < nPU; i++) total += (size_t)(desc[i].right - desc[i].left + 1) * (desc[i].bottom - desc[i].top + 1);
    memcpy(arena, desc, (size_t)nPU * sizeof(cucd_me_desc));
    const int rc = call(CUCD_IPC_ME_SURFACE, nPU, (size_t)nPU * sizeof(cucd_me_desc), total * 4);
    if (rc == CUCD_OK) memcpy(sadOut, reply(), total * 4);
    return rc;
  }
  int me_subpel_cost(int nPU, const cucd_subpel_desc* desc, uint32_t* cost) {
    memcpy(arena, desc, (size_t)nPU * sizeof(cucd_subpel_desc));
    const int rc = call(CUCD_IPC_SUBPEL, nPU, (size_t)nPU * sizeof(cucd_subpel_desc), (size_t)nPU * CUCD_SUBPEL_POINTS * 4);
    if (rc == CUCD_OK) memcpy(cost, reply(), (size_t)nPU * CUCD_SUBPEL_POINTS * 4);
    return rc;
  }
  /* cucd_me_mc_cost: reply = [dist | pad | pred]; pred may be NULL (args[0] tells the server) */
  int me_mc_cost(int nPU, const cucd_mc_desc* desc, uint32_t* dist, int16_t* pred) {
    if (nPU < 0 || (nPU > 0 && (!desc || !dist))) { snprintf(err, sizeof err, "me_mc_cost: bad argument"); return CUCD_ERR_INVALID; }
    size_t samples = 0;
    for (int i = 0; i < nPU; i++) samples += (size_t)(desc[i].w > 0 ? desc[i].w : 0) * (size_t)(desc[i].h > 0 ? desc[i].h : 0);
    const size_t inBytes = (size_t)nPU * sizeof(cucd_mc_desc), distBytes = ((size_t)nPU * 4 + 15) & ~(size_t)15;
    const size_t outBytes = distBytes + (pred ? samples * 2 : 0);
    if (((inBytes + 255) & ~(size_t)255) + outBytes > hdr->arena_bytes) {
      snprintf(err, sizeof err, "me_mc_cost: %d candidates need %llu bytes, more than the %llu-byte arena", nPU,
               (unsigned long long)(((inBytes + 255) & ~(size_t)255) + outBytes), (unsigned long long)hdr->arena_bytes);
      return CUCD_ERR_NOMEM;
    }
    memcpy(arena, desc, inBytes);
    s->args[0] = pred ? 1 : 0;
    const int rc = call(CUCD_IPC_MC, nPU, inBytes, outBytes);
    if (rc == CUCD_OK) { memcpy(dist, reply(), (size_t)nPU * 4); if (pred) memcpy(pred, reply() + distBytes, samples * 2); }
    return rc;
  }
  /* cucd_set_ref_picture_chroma: request = [padded Cb | padded Cr], (W/2 + 2 marginX) x (H/2 + 2 marginY) each, tight */
  int set_ref_picture_chroma(int W, int H, int ref_idx, const int16_t* recCb, const int16_t* recCr, int strideC, int marginX, int marginY) {
    const int pw = W / 2 + 2 * marginX, ph = H / 2 + 2 * marginY;
    const size_t plane = (size_t)pw * ph;
    const int16_t* src[2] = {recCb, recCr};
    for (int c = 0; c < 2; c++) {
      const int16_t* first = src[c] - (ptrdiff_t)marginY * strideC - marginX;
      for (int r = 0; r < ph; r++) memcpy(arena + (c * plane + (size_t)r * pw) * 2, first + (size_t)r * strideC, (size_t)pw * 2);
    }
    s->args[0] = ref_idx; s->args[1] = marginX; s->args[2] = marginY;
    return call(CUCD_IPC_SET_REF_CHROMA, 1, 2 * plane * 2, 0);
  }
  /* cucd_set_cur_picture_chroma: request = [Cb | Cr], (W/2) x (H/2) each, tight */
  int set_cur_picture_chroma(int W, int H, const int16_t* orgCb, const int16_t* orgCr, int strideC) {
    const size_t plane = (size_t)(W / 2) * (H / 2);
    const int16_t* src[2] = {orgCb, orgCr};
    for (int c = 0; c < 2; c++)
      for (int r = 0; r < H / 2; r++) memcpy(arena + (c * plane + (size_t)r * (W / 2)) * 2, src[c] + (size_t)r * strideC, (size_t)(W / 2) * 2);
    return call(CUCD_IPC_SET_CUR_CHROMA, 1, 2 * plane * 2, 0);
  }
  /* cucd_me_mc_chroma: reply = [sse (2 per candidate) | pad | pred (Cb, Cr blocks)]; pred may be NULL (args[0] tells the server) */
  int me_mc_chroma(int nPU, const cucd_mc_desc* desc, uint32_t* sse, int16_t* pred) {
    if (nPU < 0 || (nPU > 0 && (!desc || !sse))) { snprintf(err, sizeof err, "me_mc_chroma: bad argument"); return CUCD_ERR_INVALID; }
    size_t samples = 0;
    for (int i = 0; i < nPU; i++) samples += 2 * (size_t)(desc[i].w > 0 ? desc[i].w / 2 : 0) * (size_t)(desc[i].h > 0 ? desc[i].h / 2 : 0);
    const size_t inBytes = (size_t)nPU * sizeof(cucd_mc_desc), sseBytes = ((size_t)nPU * 8 + 15) & ~(size_t)15;
    const size_t outBytes = sseBytes + (pred ? samples * 2 : 0);
    if (((inBytes + 255) & ~(size_t)255) + outBytes > hdr->arena_bytes) {
      snprintf(err, sizeof err, "me_mc_chroma: %d candidates need %llu bytes, more than the %llu-byte arena", nPU,
               (unsigned long long)(((inBytes + 255) & ~(size_t)255) + outBytes), (unsigned long long)hdr->arena_bytes);
      return CUCD_ERR_NOMEM;
    }
    memcpy(arena, desc, inBytes);
    s->args[0] = pred ? 1 : 0;
    const int rc = call(CUCD_IPC_MC_CHROMA, nPU, inBytes, outBytes);
    if (rc == CUCD_OK) { memcpy(sse, reply(), (size_t)nPU * 8); if (pred) memcpy(pred, reply() + sseBytes, samples * 2); }
    return rc;
  }
  /* cucd_me_search: reply = one cucd_search_result per PU */
  int me_search(int nPU, const cucd_search_desc* desc, cucd_search_result* out) {
    if (nPU < 0 || (nPU > 0 && (!desc || !out))) { snprintf(err, sizeof err, "me_search: bad argument"); return CUCD_ERR_INVALID; }
    const size_t inBytes = (size_t)nPU * sizeof(cucd_search_desc), outBytes = (size_t)nPU * sizeof(cucd_search_result);
    if (((inBytes + 255) & ~(size_t)255) + outBytes > hdr->arena_bytes) {
      snprintf(err, sizeof err, "me_search: %d PUs need %llu bytes, more than the %llu-byte arena", nPU,
               (unsigned long long)(((inBytes + 255) & ~(size_t)255) + outBytes), (unsigned long long)hdr->arena_bytes);
      return CUCD_ERR_NOMEM;
    }
    memcpy(arena, desc, inBytes);
    const int rc = call(CUCD_IPC_ME_SEARCH, nPU, inBytes, outBytes);
    if (rc == CUCD_OK) memcpy(out, reply(), outBytes);
    return rc;
  }
  /* cucd_me_tz_search: reply = one cucd_search_result per PU */
  int me_tz_search(int nPU, const cucd_tz_desc* desc, cucd_search_result* out) {
    if (nPU < 0 || (nPU > 0 && (!desc || !out))) { snprintf(err, sizeof err, "me_tz_search: bad argument"); return CUCD_ERR_INVALID; }
    const size_t inBytes = (size_t)nPU * sizeof(cucd_tz_desc), outBytes = (size_t)nPU * sizeof(cucd_search_result);
    if (((inBytes + 255) & ~(size_t)255) + outBytes > hdr->arena_bytes) {
      snprintf(err, sizeof err, "me_tz_search: %d PUs need %llu bytes, more than the %llu-byte arena", nPU,
               (unsigned long long)(((inBytes + 255) & ~(size_t)255) + outBytes), (unsigned long long)hdr->arena_bytes);
      return CUCD_ERR_NOMEM;
    }
    memcpy(arena, desc, inBytes);
    const int rc = call(CUCD_IPC_ME_TZ_SEARCH, nPU, inBytes, outBytes);
    if (rc == CUCD_OK) memcpy(out, reply(), outBytes);
    return rc;
  }
};
#endif
