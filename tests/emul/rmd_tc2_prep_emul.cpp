// rmd_tc2_prep_emul.cpp - CPU replay of the border pre-pass of the 8-bit tensor-core RMD kernel (TEST HARNESS, not a product path).
//
// Compiles csrc/rmd_tc2.cuh and csrc/rmd_tc_frame.cuh with g++ and replays rmd_border_prep_kernel (prep_phase for every thread id
// between its barriers) and the bulk copies of tc2_prep_copies (prep_copy) as byte copies.  check_images compares the store and DC
// sums this gives an RMD CTA with the ones the CTA's own prologue built before the pre-pass existed (tile_store + build_unfiltered +
// build_filtered in the CTA, as tests/emul/rmd_tc2_emul.cpp still replays it).  Built by tests/test_tc2_border_prep.py.
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <vector>
#include "rmd_tc2.cuh"
#include "rmd_tc_frame.cuh"

using namespace cucd;
using namespace cucd::tc2;
using namespace cucd::tcf;

namespace {

// rmd_border_prep_kernel over CTUs 0 .. totalCtus-1 of fs: the images, kPrepCtuBytes per CTU
std::vector<uint8_t> emul_prep(const FrameSource& fs, int strong, int totalCtus) {
  std::vector<uint8_t> img((size_t)totalCtus * kPrepCtuBytes, 0xC3);
  std::vector<Vec16> tileBuf(Cfg<2>::TILE_BYTES / 16), stageBuf(kPrepStageBytes / 16);
  unsigned char* tile = reinterpret_cast<unsigned char*>(tileBuf.data());
  unsigned char* stage = reinterpret_cast<unsigned char*>(stageBuf.data());
  for (int cg = 0; cg < totalCtus; cg++) {
    const CtuPos pos = ctu_pos(fs, cg);
    std::memset(tile, 0x3C, Cfg<2>::TILE_BYTES);
    std::memset(stage, 0xA5, kPrepStageBytes);     // what an earlier CTA left in shared memory
    stage_tile<2>(0, 1, fs.rec + (size_t)pos.pic * fs.recPicStride, fs.recStride, fs.W, fs.H, pos.x, pos.y, tile);
    auto depth = [&](auto tag) {
      constexpr int L = decltype(tag)::value;
      int any = 0;
      for (int tid = 0; tid < kTileThreads; tid++) any |= prep_phase<L>(0, fs, strong, cg, pos, tile, tid, stage, img.data());
      if (!any) return;                            // as the kernel: nothing to evaluate, no image
      for (int ph = 1; ph < kPrepPhases; ph++)
        for (int tid = 0; tid < kTileThreads; tid++) prep_phase<L>(ph, fs, strong, cg, pos, tile, tid, stage, img.data());
    };
    depth(std::integral_constant<int, 6>());
    depth(std::integral_constant<int, 5>());
    depth(std::integral_constant<int, 4>());
    depth(std::integral_constant<int, 3>());
    depth(std::integral_constant<int, 2>());
  }
  return img;
}

// the PU states of the unit's CTUs (frame mode), as tc2_prologue writes them
template <int LOG2N>
void frame_states(const FrameSource& fs, int unit, const int* ctuXs, const int* ctuYs, uint8_t* valid) {
  for (int c = 0; c < Cfg<LOG2N>::CTUS; c++) {
    if (ctuXs[c] < 0) { for (int p = 0; p < Cfg<LOG2N>::PUS; p++) valid[c * 256 + p] = kPuOutside; continue; }
    const uint8_t* need = ctu_needed<LOG2N>(fs, unit * Cfg<LOG2N>::CTUS + c);
    for (int p = 0; p < Cfg<LOG2N>::PUS; p++) valid[c * 256 + p] = pu_state<LOG2N>(fs, need, ctuXs[c], ctuYs[c], p);
  }
}
// the bulk copies of tc2_prep_copies: the images of the unit's CTUs into the store and the DC sums
template <int LOG2N>
void place_images(const uint8_t* img, int unit, int totalCtus, unsigned char* smem) {
  for (int c = 0; c < Cfg<LOG2N>::CTUS && unit * Cfg<LOG2N>::CTUS + c < totalCtus; c++)
    for (int i = 0; i < prep_copies<LOG2N>(); i++) {
      const PrepCopy pc = prep_copy<LOG2N>(c, i);
      std::memcpy(smem + pc.dst, img + (size_t)(unit * Cfg<LOG2N>::CTUS + c) * kPrepCtuBytes + prep_off<LOG2N>() + pc.src, pc.bytes);
    }
}

// The store and DC sums of the CTA of `unit` as the in-kernel prologue built them before the border pre-pass (tile_store of each CTU's
// neighbourhood into the CTA, build_unfiltered / build_filtered on it) against the ones the pre-pass images give after place_images.
// Bytes the builders never write are found by building twice, on shared memory filled with 0x00 and with 0xFF, and not compared.
// Returns the number of differing bytes; adds the number compared to *compared.
template <int LOG2N>
long long check_images(const FrameSource& fs, int strong, int totalCtus, int unit, const uint8_t* img, long long* compared) {
  typedef Cfg<LOG2N> C;
  int ctuXs[C::CTUS], ctuYs[C::CTUS];
  Vec16 pre[8];
  setup_loads<Cfg, LOG2N>(fs, unit, totalCtus, 0, ctuXs, ctuYs, nullptr, pre);
  auto old_prologue = [&](unsigned char fill) {
    std::vector<Vec16> buf(C::TOTAL / 16), tiles(C::CTUS * C::TILE_BYTES / 16);
    unsigned char* smem = reinterpret_cast<unsigned char*>(buf.data());
    unsigned char* t = reinterpret_cast<unsigned char*>(tiles.data());
    std::memset(smem, fill, C::TOTAL);
    for (int i = 0; i < C::CTUS * 64; i++) reinterpret_cast<int*>(smem + C::DC_OFF)[i] = 0;
    frame_states<LOG2N>(fs, unit, ctuXs, ctuYs, smem + C::VALID_OFF);
    for (int c = 0; c < C::CTUS; c++)
      if (ctuXs[c] >= 0) stage_tile<LOG2N>(0, 1, fs.rec + (size_t)ctu_pos(fs, unit * C::CTUS + c).pic * fs.recPicStride, fs.recStride, fs.W, fs.H, ctuXs[c], ctuYs[c], t + c * C::TILE_BYTES);
    for (int c = 0; c < C::CTUS; c++)
      if (ctuXs[c] >= 0) for (int tid = 0; tid < kThreads; tid++) build_unfiltered<LOG2N>(tid, c, fs.W, fs.H, ctuXs[c], ctuYs[c], t + c * C::TILE_BYTES, smem);
    for (int c = 0; c < C::CTUS; c++)
      if (ctuXs[c] >= 0) for (int tid = 0; tid < kThreads; tid++) build_filtered<LOG2N>(tid, c, strong, smem);
    return buf;
  };
  const std::vector<Vec16> b0 = old_prologue(0x00), b1 = old_prologue(0xFF);
  std::vector<Vec16> bn(C::TOTAL / 16);
  unsigned char* sn = reinterpret_cast<unsigned char*>(bn.data());
  std::memset(sn, 0x5A, C::TOTAL);
  frame_states<LOG2N>(fs, unit, ctuXs, ctuYs, sn + C::VALID_OFF);
  place_images<LOG2N>(img, unit, totalCtus, sn);
  const unsigned char* s0 = reinterpret_cast<const unsigned char*>(b0.data());
  const unsigned char* s1 = reinterpret_cast<const unsigned char*>(b1.data());
  long long bad = 0;
  for (int i = C::STORE_OFF; i < C::STORE_OFF + C::STORE_BYTES; i++) {
    if (s0[i] != s1[i]) continue;
    ++*compared;
    bad += sn[i] != s0[i];
  }
  for (int c = 0; c < C::CTUS; c++) {
    if (ctuXs[c] < 0 || LOG2N == 2) continue;
    for (int p = 0; p < C::PUS; p++) {
      if (sn[C::VALID_OFF + c * 256 + p] != kPuEvaluate) continue;   // read by dc_tile of an evaluated PU only
      const int o = C::DC_OFF + (c * 64 + p) * 4;
      *compared += 4;
      bad += std::memcmp(sn + o, s0 + o, 4) != 0;
    }
  }
  return bad;
}

FrameSource picture_source(const int16_t* org, int orgStride, const int16_t* rec, int recStride, int W, int H, uint32_t* out, const uint8_t* needed) {
  FrameSource fs;
  fs.org = org; fs.rec = rec; fs.orgPicStride = 0; fs.recPicStride = 0; fs.orgStride = orgStride; fs.recStride = recStride;
  fs.W = W; fs.H = H; fs.ctusPerRow = (W + 63) / 64; fs.ctusPerPic = fs.ctusPerRow * ((H + 63) / 64); fs.out = out; fs.outPacked = nullptr; fs.needed = needed;
  return fs;
}

}  // namespace

extern "C" {

// border pre-pass of one picture: img[ctus * emul_tc2_prep_ctu_bytes()]
int emul_tc2_prep_ctu_bytes() { return kPrepCtuBytes; }
int emul_tc2_prep_images(int strong, const int16_t* rec, int recStride, int W, int H, uint8_t* img) {
  const FrameSource fs = picture_source(rec, recStride, rec, recStride, W, H, nullptr, nullptr);
  const std::vector<uint8_t> v = emul_prep(fs, strong, fs.ctusPerPic);
  std::memcpy(img, v.data(), v.size());
  return 0;
}
// check_images over every CTA of one picture at every depth: differing bytes (*compared: bytes compared)
long long emul_tc2_prep_check(int strong, const int16_t* rec, int recStride, int W, int H, long long* compared) {
  const FrameSource fs = picture_source(rec, recStride, rec, recStride, W, H, nullptr, nullptr);
  const int total = fs.ctusPerPic;
  const std::vector<uint8_t> img = emul_prep(fs, strong, total);
  long long bad = 0;
  *compared = 0;
  for (int b = 0; b < frame_blocks(total); b++) {
    const FrameBlock fb = frame_block(total, b);
    switch (fb.log2n) {
      case 6: bad += check_images<6>(fs, strong, total, fb.unit, img.data(), compared); break;
      case 5: bad += check_images<5>(fs, strong, total, fb.unit, img.data(), compared); break;
      case 4: bad += check_images<4>(fs, strong, total, fb.unit, img.data(), compared); break;
      case 3: bad += check_images<3>(fs, strong, total, fb.unit, img.data(), compared); break;
      default: bad += check_images<2>(fs, strong, total, fb.unit, img.data(), compared);
    }
  }
  return bad;
}
}  // extern "C"
