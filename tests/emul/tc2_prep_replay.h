// tc2_prep_replay.h - CPU replay of the border pre-pass of the 8-bit tensor-core RMD kernel (TEST HARNESS, not a product path).
//
// rmd_border_prep_kernel (prep_phase for every thread id between its barriers) and the bulk copies of tc2_prep_copies (prep_copy) as
// byte copies.  Shared by tests/emul/rmd_tc2_emul.cpp (the RMD CTA replayed on the images, as the GPU runs it) and
// tests/emul/rmd_tc2_prep_emul.cpp (the images against the CTA's own prologue).  Include after rmd_tc2.cuh and rmd_tc_frame.cuh.
#pragma once
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <vector>
#include "rmd_tc2.cuh"
#include "rmd_tc_frame.cuh"

namespace cucd {
namespace tc2replay {

// rmd_border_prep_kernel over CTUs 0 .. totalCtus-1 of fs (fs.needed: the fork-aware mask or null): the images, kPrepCtuBytes per CTU.
// The buffer starts as `poison` everywhere, as a scratch an earlier launch left: a (CTU, depth) the kernel writes no image for keeps it.
inline std::vector<uint8_t> emul_prep(const FrameSource& fs, int strong, int totalCtus, uint8_t poison = 0xC3) {
  using namespace cucd::tc2;
  using namespace cucd::tcf;
  std::vector<uint8_t> img((size_t)totalCtus * kPrepCtuBytes, poison);
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

// the bulk copies of tc2_prep_copies: the images of the unit's CTUs into the store and the DC sums of the CTA's shared memory
template <int LOG2N>
void place_images(const uint8_t* img, int unit, int totalCtus, unsigned char* smem) {
  using namespace cucd::tc2;
  for (int c = 0; c < Cfg<LOG2N>::CTUS && unit * Cfg<LOG2N>::CTUS + c < totalCtus; c++)
    for (int i = 0; i < prep_copies<LOG2N>(); i++) {
      const PrepCopy pc = prep_copy<LOG2N>(c, i);
      std::memcpy(smem + pc.dst, img + (size_t)(unit * Cfg<LOG2N>::CTUS + c) * kPrepCtuBytes + prep_off<LOG2N>() + pc.src, pc.bytes);
    }
}

}  // namespace tc2replay
}  // namespace cucd
