// ipc_replay NAME JOB OUT: one client process of cucd_server (include/cucd_ipc.h) for tests/test_gpu_encoder_workloads.py.
// JOB holds int32 W, H, bitDepth, nPics, nPU, orgN, brdN, nMe, nSp, margin, then the nPics int16 luma planes, nPU int32 log2
// sizes, the PUs' int16 source blocks and borders back to back, and - when nMe > 0 - the int16 padded reference plane, nMe
// cucd_me_desc and nSp cucd_subpel_desc.  The client sends what an encoder instance sends: one cuCUDecide_frame per picture, one
// single-PU cucd_intra_rmd_batch per PU, and (picture 1 against the reference) per PU an ME surface and a sub-pel table.
// OUT receives every reply in that order.
#include <vector>
#include "cucd_ipc.h"

int main(int argc, char** argv) {
  if (argc != 4) { fprintf(stderr, "usage: ipc_replay NAME JOB OUT\n"); return 2; }
  FILE* f = fopen(argv[2], "rb");
  if (!f) { perror(argv[2]); return 2; }
  int32_t h[10];
  if (fread(h, 4, 10, f) != 10) return 2;
  const int W = h[0], H = h[1], bd = h[2], nPics = h[3], nPU = h[4], nMe = h[7], nSp = h[8], margin = h[9];
  auto rd = [&](auto& v, size_t n) { v.resize(n); return fread(v.data(), sizeof(v[0]), n, f) == n; };
  std::vector<int16_t> pics, org, brd, ref;
  std::vector<int32_t> log2s;
  std::vector<cucd_me_desc> me;
  std::vector<cucd_subpel_desc> sp;
  if (!rd(pics, (size_t)nPics * W * H) || !rd(log2s, nPU) || !rd(org, h[5]) || !rd(brd, h[6]) ||
      (nMe && !rd(ref, (size_t)(W + 2 * margin) * (H + 2 * margin))) || !rd(me, nMe) || !rd(sp, nSp)) { fprintf(stderr, "short job file\n"); return 2; }
  fclose(f);
  FILE* out = fopen(argv[3], "wb");
  cucd_ipc_client c;
  auto check = [&](int rc, const char* what) { if (rc != CUCD_OK) { fprintf(stderr, "%s: %d %s\n", what, rc, c.err); exit(1); } };
  check(c.connect(argv[1]), "connect");
  check(c.open(W, H, bd, 1), "open");
  std::vector<int16_t> obf((size_t)(W / 4) * (H / 4)), outl((size_t)W * H);
  for (int p = 0; p < nPics; p++) {
    check(c.frame(W, H, pics.data() + (size_t)p * W * H, W, obf.data(), outl.data()), "frame");
    fwrite(obf.data(), 2, obf.size(), out); fwrite(outl.data(), 2, outl.size(), out);
  }
  size_t oo = 0, bo = 0;
  for (int i = 0; i < nPU; i++) {
    cucd_pu_desc d = {};
    d.log2_size = (uint8_t)log2s[i];
    uint32_t sad[35];
    check(c.intra_rmd_batch(1, &d, org.data() + oo, brd.data() + bo, sad), "rmd");
    fwrite(sad, 4, 35, out);
    oo += (size_t)1 << (2 * log2s[i]); bo += ((size_t)4 << log2s[i]) + 1;
  }
  if (nMe) {
    check(c.set_cur_picture(W, H, pics.data() + (size_t)W * H, W), "set_cur");
    check(c.set_ref_picture(W, H, 0, ref.data() + (size_t)margin * (W + 2 * margin) + margin, W + 2 * margin, margin, margin), "set_ref");
  }
  for (int i = 0; i < nMe; i++) {
    std::vector<uint32_t> s((size_t)(me[i].right - me[i].left + 1) * (me[i].bottom - me[i].top + 1));
    check(c.me_sad_surface(1, &me[i], s.data()), "me_sad_surface");
    fwrite(s.data(), 4, s.size(), out);
    uint32_t t[CUCD_SUBPEL_POINTS];
    check(c.me_subpel_cost(1, &sp[i], t), "me_subpel_cost");
    fwrite(t, 4, CUCD_SUBPEL_POINTS, out);
  }
  c.close_client();
  fclose(out);
  return 0;
}
