// ipc_me_tz_replay NAME JOB OUT: one client process of cucd_server (include/cucd_ipc.h) for tests/test_gpu_me_tz_search.py.
// JOB holds int32 W, H, bitDepth, margin, nRef, nP, then nRef int32 slots, the int16 source plane (W x H), the nRef int16 padded
// reference planes ((W + 2 margin) x (H + 2 margin) each) and nP cucd_tz_desc.  The client sends set-cur, one set-ref per slot,
// one cucd_me_tz_search request with all PUs, then one request per PU.  OUT receives the results of the first request, then those
// of every single-PU request.
#include <vector>
#include "cucd_ipc.h"

int main(int argc, char** argv) {
  if (argc != 4) { fprintf(stderr, "usage: ipc_me_tz_replay NAME JOB OUT\n"); return 2; }
  FILE* f = fopen(argv[2], "rb");
  if (!f) { perror(argv[2]); return 2; }
  int32_t h[6];
  if (fread(h, 4, 6, f) != 6) return 2;
  const int W = h[0], H = h[1], bd = h[2], margin = h[3], nRef = h[4], nP = h[5];
  const int pw = W + 2 * margin, ph = H + 2 * margin;
  auto rd = [&](auto& v, size_t n) { v.resize(n); return fread(v.data(), sizeof(v[0]), n, f) == n; };
  std::vector<int32_t> slots;
  std::vector<int16_t> cur, refs;
  std::vector<cucd_tz_desc> desc;
  if (!rd(slots, nRef) || !rd(cur, (size_t)W * H) || !rd(refs, (size_t)nRef * pw * ph) || !rd(desc, nP)) { fprintf(stderr, "short job file\n"); return 2; }
  fclose(f);
  FILE* out = fopen(argv[3], "wb");
  cucd_ipc_client c;
  auto check = [&](int rc, const char* what) { if (rc != CUCD_OK) { fprintf(stderr, "%s: %d %s\n", what, rc, c.err); exit(1); } };
  check(c.connect(argv[1]), "connect");
  check(c.open(W, H, bd, 1), "open");
  check(c.set_cur_picture(W, H, cur.data(), W), "set_cur");
  for (int r = 0; r < nRef; r++)
    check(c.set_ref_picture(W, H, slots[r], refs.data() + (size_t)r * pw * ph + (size_t)margin * pw + margin, pw, margin, margin), "set_ref");
  std::vector<cucd_search_result> res(nP);
  check(c.me_tz_search(nP, desc.data(), res.data()), "me_tz_search");
  fwrite(res.data(), sizeof(cucd_search_result), res.size(), out);
  for (int i = 0; i < nP; i++) {
    cucd_search_result r1;
    check(c.me_tz_search(1, &desc[i], &r1), "me_tz_search single");
    fwrite(&r1, sizeof r1, 1, out);
  }
  c.close_client();
  fclose(out);
  return 0;
}
