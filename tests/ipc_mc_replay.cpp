// ipc_mc_replay NAME JOB OUT: one client process of cucd_server (include/cucd_ipc.h) for tests/test_gpu_mc.py.
// JOB holds int32 W, H, bitDepth, margin, nRef, nC, then nRef int32 slots, the int16 source plane (W x H), the nRef int16 padded
// reference planes ((W + 2 margin) x (H + 2 margin) each) and nC cucd_mc_desc.  The client sends set-cur, one set-ref per slot, one
// cucd_me_mc_cost request with all candidates and predictions, one without predictions, then one request per candidate.
// OUT receives dist + pred of the first request, dist of the second, then dist + pred of every single-candidate request.
#include <vector>
#include "cucd_ipc.h"

int main(int argc, char** argv) {
  if (argc != 4) { fprintf(stderr, "usage: ipc_mc_replay NAME JOB OUT\n"); return 2; }
  FILE* f = fopen(argv[2], "rb");
  if (!f) { perror(argv[2]); return 2; }
  int32_t h[6];
  if (fread(h, 4, 6, f) != 6) return 2;
  const int W = h[0], H = h[1], bd = h[2], margin = h[3], nRef = h[4], nC = h[5];
  const int pw = W + 2 * margin, ph = H + 2 * margin;
  auto rd = [&](auto& v, size_t n) { v.resize(n); return fread(v.data(), sizeof(v[0]), n, f) == n; };
  std::vector<int32_t> slots;
  std::vector<int16_t> cur, refs;
  std::vector<cucd_mc_desc> desc;
  if (!rd(slots, nRef) || !rd(cur, (size_t)W * H) || !rd(refs, (size_t)nRef * pw * ph) || !rd(desc, nC)) { fprintf(stderr, "short job file\n"); return 2; }
  fclose(f);
  size_t samples = 0;
  for (const cucd_mc_desc& d : desc) samples += (size_t)d.w * d.h;
  FILE* out = fopen(argv[3], "wb");
  cucd_ipc_client c;
  auto check = [&](int rc, const char* what) { if (rc != CUCD_OK) { fprintf(stderr, "%s: %d %s\n", what, rc, c.err); exit(1); } };
  check(c.connect(argv[1]), "connect");
  check(c.open(W, H, bd, 1), "open");
  check(c.set_cur_picture(W, H, cur.data(), W), "set_cur");
  for (int r = 0; r < nRef; r++)
    check(c.set_ref_picture(W, H, slots[r], refs.data() + (size_t)r * pw * ph + (size_t)margin * pw + margin, pw, margin, margin), "set_ref");
  std::vector<uint32_t> dist(nC);
  std::vector<int16_t> pred(samples);
  check(c.me_mc_cost(nC, desc.data(), dist.data(), pred.data()), "me_mc_cost");
  fwrite(dist.data(), 4, dist.size(), out); fwrite(pred.data(), 2, pred.size(), out);
  check(c.me_mc_cost(nC, desc.data(), dist.data(), nullptr), "me_mc_cost without pred");
  fwrite(dist.data(), 4, dist.size(), out);
  for (int i = 0; i < nC; i++) {
    uint32_t d1;
    std::vector<int16_t> p1((size_t)desc[i].w * desc[i].h);
    check(c.me_mc_cost(1, &desc[i], &d1, p1.data()), "me_mc_cost single");
    fwrite(&d1, 4, 1, out); fwrite(p1.data(), 2, p1.size(), out);
  }
  c.close_client();
  fclose(out);
  return 0;
}
