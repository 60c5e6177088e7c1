// ipc_mc_chroma_replay NAME JOB OUT: one client process of cucd_server (include/cucd_ipc.h) for tests/test_gpu_mc_chroma.py.
// JOB holds int32 W, H, bitDepth, margin, nRef, nC, then nRef int32 slots, the int16 source planes (luma W x H, then Cb and Cr,
// W/2 x H/2 each), per slot the padded luma plane ((W + 2 margin) x (H + 2 margin)) and the padded Cb and Cr planes (margin / 2), and
// nC cucd_mc_desc.  The client sends set-cur and set-cur-chroma, set-ref and set-ref-chroma per slot, one cucd_me_mc_chroma request with
// all candidates and predictions, one without predictions, then one request per candidate.
// OUT receives sse + pred of the first request, sse of the second, then sse + pred of every single-candidate request.
#include <vector>
#include "cucd_ipc.h"

int main(int argc, char** argv) {
  if (argc != 4) { fprintf(stderr, "usage: ipc_mc_chroma_replay NAME JOB OUT\n"); return 2; }
  FILE* f = fopen(argv[2], "rb");
  if (!f) { perror(argv[2]); return 2; }
  int32_t h[6];
  if (fread(h, 4, 6, f) != 6) return 2;
  const int W = h[0], H = h[1], bd = h[2], margin = h[3], nRef = h[4], nC = h[5];
  const int mc = margin / 2, pw = W + 2 * margin, ph = H + 2 * margin, pwc = W / 2 + 2 * mc, phc = H / 2 + 2 * mc;
  const size_t lumaRef = (size_t)pw * ph, chromaRef = (size_t)pwc * phc, chroma = (size_t)(W / 2) * (H / 2);
  auto rd = [&](auto& v, size_t n) { v.resize(n); return fread(v.data(), sizeof(v[0]), n, f) == n; };
  std::vector<int32_t> slots;
  std::vector<int16_t> cur, curC, refs;
  std::vector<cucd_mc_desc> desc;
  if (!rd(slots, nRef) || !rd(cur, (size_t)W * H) || !rd(curC, 2 * chroma) || !rd(refs, (size_t)nRef * (lumaRef + 2 * chromaRef)) || !rd(desc, nC)) {
    fprintf(stderr, "short job file\n");
    return 2;
  }
  fclose(f);
  size_t samples = 0;
  for (const cucd_mc_desc& d : desc) samples += 2 * (size_t)(d.w / 2) * (d.h / 2);
  FILE* out = fopen(argv[3], "wb");
  cucd_ipc_client c;
  auto check = [&](int rc, const char* what) { if (rc != CUCD_OK) { fprintf(stderr, "%s: %d %s\n", what, rc, c.err); exit(1); } };
  check(c.connect(argv[1]), "connect");
  check(c.open(W, H, bd, 1), "open");
  check(c.set_cur_picture(W, H, cur.data(), W), "set_cur");
  check(c.set_cur_picture_chroma(W, H, curC.data(), curC.data() + chroma, W / 2), "set_cur_chroma");
  for (int r = 0; r < nRef; r++) {
    const int16_t* base = refs.data() + (size_t)r * (lumaRef + 2 * chromaRef);
    check(c.set_ref_picture(W, H, slots[r], base + (size_t)margin * pw + margin, pw, margin, margin), "set_ref");
    const int16_t* cb = base + lumaRef + (size_t)mc * pwc + mc;
    check(c.set_ref_picture_chroma(W, H, slots[r], cb, cb + chromaRef, pwc, mc, mc), "set_ref_chroma");
  }
  std::vector<uint32_t> sse(2 * (size_t)nC);
  std::vector<int16_t> pred(samples);
  check(c.me_mc_chroma(nC, desc.data(), sse.data(), pred.data()), "me_mc_chroma");
  fwrite(sse.data(), 4, sse.size(), out); fwrite(pred.data(), 2, pred.size(), out);
  check(c.me_mc_chroma(nC, desc.data(), sse.data(), nullptr), "me_mc_chroma without pred");
  fwrite(sse.data(), 4, sse.size(), out);
  for (int i = 0; i < nC; i++) {
    uint32_t s1[2];
    std::vector<int16_t> p1(2 * (size_t)(desc[i].w / 2) * (desc[i].h / 2));
    check(c.me_mc_chroma(1, &desc[i], s1, p1.data()), "me_mc_chroma single");
    fwrite(s1, 4, 2, out); fwrite(p1.data(), 2, p1.size(), out);
  }
  c.close_client();
  fclose(out);
  return 0;
}
