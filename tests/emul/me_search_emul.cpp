// me_search_emul.cpp - CPU replay of the motion-search phases of cucd_me_search (TEST HARNESS, not a product path).
//
// The Argmin form of the SAD kernels (csrc/me_kernels.cu) ends every thread's candidates in a search key and reduces the keys of a
// warp with a 64-bit xor butterfly before one atomicMin per warp; the prep and walk kernels are one thread per PU / per FRAC PU around
// me_search_prep / me_search_walk (csrc/me_core.cuh).  This file replays, for every thread id:
//   emul_me_search_key   the tiles of one window: dy-lane tiles (M / E) with their own SAD arithmetic (me_dy_*) and key
//                        (me_dy_lane_key); dx-lane tiles (O) with the SAD of the caller's surface at the lane's candidate(s), the
//                        thread layout of me_sad_kernel (32 x 8, one candidate) or me_sad_u8_kernel (32 x 16, dy and dy + 8);
//                        then the warp butterfly and the atomicMin of every warp
//   emul_me_search_prep  me_search_prep for every PU
//   emul_me_search_walk  me_search_walk for one PU
#include <cstdint>
#include <cstring>
#include <vector>
#include "me_core.cuh"

using namespace cucd;

namespace {

// field for field the layouts of MeJob / SubpelJob (csrc/kernels.h), which me_search_prep takes as template arguments
struct Job { int32_t curOff, refOff, refSlot; int16_t w, h, left, right, top, bottom, subShift, pad; int64_t outOff; };
struct Sub { int32_t curOff, refOff, refSlot; int16_t w, h; int32_t useHadamard; };

// me_key_warp_commit: xor butterfly over the 32 lanes, then lane 0's atomicMin
void warp_commit(unsigned long long* lanes, unsigned long long* key) {
  for (int m = 16; m > 0; m >>= 1) {
    unsigned long long next[32];
    for (int l = 0; l < 32; l++) next[l] = me_key_min(lanes[l], lanes[l ^ m]);
    std::memcpy(lanes, next, sizeof(next));
  }
  if (lanes[0] != kMeNoKey && lanes[0] < *key) *key = lanes[0];
}

template <bool U8>
void replay_dy_tile(int kind, int x0, int y0, int bitDepth, const int16_t* cur, int curStride, int w, int h, const int16_t* refWin, int refStride,
                    int cols, int rows, int subShift, int left, int top, const MeSearchCost& c, unsigned long long* key) {
  constexpr int P = U8 ? kMeDyPitch8 : kMeDyPitch16, SPW = U8 ? 4 : 2;
  std::vector<uint32_t> sCur(64 * 64 / SPW, 0xA5A5A5A5u), sRef((size_t)kMeDyRows * P, 0xA5A5A5A5u);
  const int step = 1 << subShift;
  const MeDyTile tl = me_dy_tile(kind, x0, y0, w, h, cols, rows);
  for (int warp = 0; warp < 8; warp++)
    for (int lane = 0; lane < 32; lane++) {
      me_dy_stage_cur<U8>(warp, lane, cur, curStride, w, h, step, sCur.data());
      me_dy_stage_ref<U8>(warp, lane, refWin + (long long)y0 * refStride + x0, refStride, tl.winW, tl.winH, sRef.data());
    }
  const int shiftOut = U8 ? 0 : bitDepth - 8;
  for (int warp = 0; warp < 8; warp++) {
    const MeDyWarp q = me_dy_warp<U8>(kind, warp, tl.cr);
    if (!(q.active && 32 * q.blk < tl.nLam)) continue;                // warp uniform: the whole warp leaves
    unsigned long long lanes[32];
    for (int lane = 0; lane < 32; lane++) {
      const int lam = 32 * q.blk + lane;
      uint32_t sad[kMeDyK];
      if (kind == kMeKindM) {
        if (U8) me_dy_sad_u8<kMeDyK>(sCur.data(), sRef.data(), w >> 2, h, step, lam, q.wbase, q.s, sad);
        else me_dy_sad_s16<kMeDyK>(sCur.data(), sRef.data(), w >> 1, h, step, lam, q.wbase, q.s, me_fold_rows(bitDepth, w >> 1), sad);
        lanes[lane] = me_dy_lane_key<kMeDyK, SPW>(sad, subShift, shiftOut, lam < tl.nLam, x0 + q.delta0, y0 + lam, cols, left, top, c);
      } else {
        if (U8) me_dy_sad_u8<1>(sCur.data(), sRef.data(), w >> 2, h, step, lam, q.wbase, q.s, sad);
        else me_dy_sad_s16<1>(sCur.data(), sRef.data(), w >> 1, h, step, lam, q.wbase, q.s, me_fold_rows(bitDepth, w >> 1), sad);
        lanes[lane] = me_dy_lane_key<1, SPW>(sad, subShift, shiftOut, lam < tl.nLam, x0 + q.delta0, y0 + lam, cols, left, top, c);
      }
    }
    warp_commit(lanes, key);
  }
}

}  // namespace

extern "C" {

// One PU.  refWin: the reference sample at the window's (left, top) displacement of the PU origin; surface[rows * cols]: the SADs the
// dx-lane tiles read (the oracle's); fast: the dy-lane kernel may run (picture-resident source and one of HM's widths); kernelO: 0
// me_sad_kernel (32 x 8), 1 me_sad_u8_kernel (32 x 16).  counts[3] = number of O / M / E tiles.  Returns keys[job] after every warp.
unsigned long long emul_me_search_key(int bitDepth, const int16_t* cur, int curStride, int w, int h, const int16_t* refWin, int refStride, int left, int right,
                                      int top, int bottom, int subShift, int fast, int kernelO, const uint32_t* surface, uint32_t lambda, int predX, int predY,
                                      int* counts) {
  const int cols = right - left + 1, rows = bottom - top + 1;
  const int tileRowsO = kernelO ? 16 : 8;
  const MeSearchCost c{lambda, predX, predY, -1};
  unsigned long long key = kMeNoKey;                                   // cudaMemsetAsync(keys, 0xff)
  counts[0] = counts[1] = counts[2] = 0;
  me_enum_tiles(cols, rows, fast != 0, tileRowsO, [&](int kind, int x0, int y0) {
    int k2, xx, yy;
    me_tile_unpack(me_tile_pack(kind, x0, y0), k2, xx, yy);
    counts[k2]++;
    if (k2 != kMeKindO) {
      if (bitDepth == 8) replay_dy_tile<true>(k2, xx, yy, bitDepth, cur, curStride, w, h, refWin, refStride, cols, rows, subShift, left, top, c, &key);
      else replay_dy_tile<false>(k2, xx, yy, bitDepth, cur, curStride, w, h, refWin, refStride, cols, rows, subShift, left, top, c, &key);
      return;
    }
    for (int warp = 0; warp < 8; warp++) {                             // every lane joins the reduction, also past the window
      unsigned long long lanes[32];
      for (int lane = 0; lane < 32; lane++) {
        const int dx = xx + lane, dyA = yy + warp;
        const bool okA = dx < cols && dyA < rows;
        unsigned long long k = okA ? me_search_key(surface[(size_t)dyA * cols + dx], dx, dyA, cols, left, top, c) : kMeNoKey;
        if (kernelO) {
          const int dyB = dyA + 8;
          const bool okB = okA && dyB < rows;
          k = me_key_min(k, okB ? me_search_key(surface[(size_t)dyB * cols + dx], dx, dyB, cols, left, top, c) : kMeNoKey);
        }
        lanes[lane] = k;
      }
      warp_commit(lanes, &key);
    }
  });
  return key;
}

// me_search_prep for i = 0 .. n - 1.  job[n][5] = (left, right, top, bottom, refOff of the PU origin), cost[n][4] = (lambda, predX,
// predY, frac), refStride of slot 0; sub jobs [nFrac]: refOffIn -> refOffOut; out[n][6] = cucd_search_result
void emul_me_search_prep(int n, const unsigned long long* keys, const int32_t* job, const int32_t* cost, int refStride, int nFrac, const int32_t* refOffIn,
                         int32_t* refOffOut, int32_t* out) {
  std::vector<Job> jobs(n);
  std::vector<MeSearchCost> costs(n);
  std::vector<Sub> subIn(nFrac > 0 ? nFrac : 1), subOut(nFrac > 0 ? nFrac : 1);
  for (int i = 0; i < n; i++) {
    Job& j = jobs[i];
    std::memset(&j, 0, sizeof(j));
    j.left = (int16_t)job[5 * i]; j.right = (int16_t)job[5 * i + 1]; j.top = (int16_t)job[5 * i + 2]; j.bottom = (int16_t)job[5 * i + 3]; j.refOff = job[5 * i + 4];
    costs[i] = MeSearchCost{(uint32_t)cost[4 * i], cost[4 * i + 1], cost[4 * i + 2], cost[4 * i + 3]};
  }
  for (int f = 0; f < nFrac; f++) { std::memset(&subIn[f], 0x5a, sizeof(Sub)); subIn[f].refSlot = 0; subIn[f].refOff = refOffIn[f]; subOut[f] = subIn[f]; subOut[f].refOff = -1; }
  const int32_t strides[1] = {refStride};
  std::vector<MeSearchOut> o(n);
  for (int i = 0; i < n; i++) me_search_prep(i, keys, jobs.data(), costs.data(), strides, subIn.data(), subOut.data(), o.data());
  std::memcpy(out, o.data(), (size_t)n * sizeof(MeSearchOut));
  for (int f = 0; f < nFrac; f++) refOffOut[f] = subOut[f].refOff;
}

// me_search_walk for one PU: res[6] holds the prep's result on entry (mvx, mvy used) and the walk's on return
void emul_me_search_walk(const uint32_t* T, uint32_t lambda, int predX, int predY, int32_t* res) {
  MeSearchOut o;
  std::memcpy(&o, res, sizeof(o));
  me_search_walk(T, MeSearchCost{lambda, predX, predY, 0}, o);
  std::memcpy(res, &o, sizeof(o));
}

}  // extern "C"
