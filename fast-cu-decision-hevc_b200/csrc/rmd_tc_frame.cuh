// rmd_tc_frame.cuh - frame-mode pieces shared by the two tensor-core RMD kernels (rmd_tc2_kernels.cu: 8-bit content,
// rmd_tc3_kernels.cu: 9/10-bit content) and by their CPU replays (tests/emul): block decode, CTU origins, PU states, the set-up
// loads of the reconstruction neighbourhoods and source tiles, the border pre-pass of the 8-bit kernel, and the copy-out of the cost
// tables.  Phase 1 of the prologue
// (TileLoad / tile_load / tile_store) is in rmd_tc2.cuh beside the border builders that read its tiles.
//
// Everything is `__host__ __device__` and holds no barrier: a function is driven per thread by (tid, nthreads), the kernel bodies
// keep their barriers between the calls (tc2 syncs its 256 workers with bar.sync 1 while its issuing warps run apart, tc3 the whole
// CTA).  Where the two kernels' shared-memory layouts differ a function takes the kernel's Cfg (tc2::Cfg or tc3::Cfg).
#pragma once
#include "rmd_tc2.cuh"

namespace cucd {
namespace tcf {

using tc2::Row;
using tc2::row_map;

using tc2::Vec16;
using tc2::TileLoad;
using tc2::tile_load;
using tc2::tile_store;

// ---------------------------------------------------------------------------------------------
// blocks of a frame launch: depth-major (as rmd_frame_kernel), a depth has ceil(totalCtus / CTUS) units of CTUS CTUs
// (Cfg::CTUS = 4 for N >= 32, 2 below)
// ---------------------------------------------------------------------------------------------
struct FrameBlock { int log2n, unit; };
CUCD_HD FrameBlock frame_block(int totalCtus, int b) {
  const int u2 = (totalCtus + 1) >> 1, u4 = (totalCtus + 3) >> 2;
  if (b < u4) return {6, b};
  b -= u4;
  if (b < u4) return {5, b};
  b -= u4;
  if (b < u2) return {4, b};
  b -= u2;
  if (b < u2) return {3, b};
  return {2, b - u2};
}
CUCD_HD int frame_blocks(int totalCtus) { return 2 * ((totalCtus + 3) >> 2) + 3 * ((totalCtus + 1) >> 1); }

// picture and sample origin of CTU cg (the CTUs of all pictures of a launch in raster order)
struct CtuPos { int pic, x, y; };
CUCD_HD CtuPos ctu_pos(const FrameSource& fs, int cg) {
  const int pic = cg / fs.ctusPerPic, ctu = cg - pic * fs.ctusPerPic;
  return {pic, (ctu % fs.ctusPerRow) * 64, (ctu / fs.ctusPerRow) * 64};
}

// first sample of the source tile of row r in CTU cg (tile origin inside the CTU from the row map); (tileX, tileY): its position
template <int LOG2N>
CUCD_HD const int16_t* frame_src_ptr(const FrameSource& fs, const Row& r, int cg, int& tileX, int& tileY) {
  constexpr int N = 1 << LOG2N;
  const CtuPos c = ctu_pos(fs, cg);
  int px, py; demorton(r.pu, px, py);
  if (LOG2N == 2) { px *= 8; py *= 8; }
  else { px = px * N + (r.o ? r.v0 : r.u0); py = py * N + (r.o ? r.u0 : r.v0); }
  tileX = c.x + px; tileY = c.y + py;
  return fs.org + (size_t)c.pic * fs.orgPicStride + (size_t)tileY * fs.orgStride + tileX;
}

// fork-aware mask of CTU cg at this depth (entry p: PU p must be evaluated), or null: every PU inside the picture is evaluated
template <int LOG2N>
CUCD_HD const uint8_t* ctu_needed(const FrameSource& fs, int cg) {
  return fs.needed ? fs.needed + ((size_t)cg * kPusPerCtu + pu_offset_of_depth(6 - LOG2N)) : nullptr;
}
// state of PU p (z order) of the CTU at (ctuX, ctuY) with mask `need`: outside the picture, pruned, or to be evaluated
template <int LOG2N>
CUCD_HD uint8_t pu_state(const FrameSource& fs, const uint8_t* need, int ctuX, int ctuY, int p) {
  constexpr int N = 1 << LOG2N;
  int px, py; demorton(p, px, py);
  const bool inside = (ctuX + (px + 1) * N <= fs.W) && (ctuY + (py + 1) * N <= fs.H);
  return !inside ? kPuOutside : ((need && !need[p]) ? kPuPruned : kPuEvaluate);
}

// Fork-aware mode, before anything else: the states of the unit's PUs into valid[c * 256 + p].  Returns whether this thread found
// a PU to evaluate; a CTA where no thread did writes the table codes (copy_out) and leaves.
template <template <int> class Cfg, int LOG2N>
CUCD_HD int fork_states(const FrameSource& fs, int unit, int totalCtus, uint8_t* valid, int tid, int nthreads) {
  typedef Cfg<LOG2N> C;
  int any = 0;
  for (int i = tid; i < C::CTUS * C::PUS; i += nthreads) {
    const int c = i / C::PUS, p = i - c * C::PUS, cg = unit * C::CTUS + c;
    if (cg >= totalCtus) continue;
    const CtuPos pos = ctu_pos(fs, cg);
    const uint8_t st = pu_state<LOG2N>(fs, ctu_needed<LOG2N>(fs, cg), pos.x, pos.y, p);
    valid[c * 256 + p] = st;
    any |= st == kPuEvaluate;
  }
  return any;
}

// The set-up loads of a CTA: the origins of the unit's CTUs (-1 past the last CTU), thread tid's part of their reconstruction
// neighbourhoods (tl; null for tc2, whose border pre-pass has read them), and `pre`, the eight rows of the source tile of the thread's
// row in pass 0 (zero unless the tile is inside the picture).
template <template <int> class Cfg, int LOG2N>
CUCD_HD void setup_loads(const FrameSource& fs, int unit, int totalCtus, int tid, int* ctuX, int* ctuY, TileLoad* tl, Vec16* pre) {
  typedef Cfg<LOG2N> C;
#pragma unroll
  for (int c = 0; c < C::CTUS; c++) {
    const int cg = unit * C::CTUS + c;
    ctuX[c] = -1; ctuY[c] = -1;
    if (cg >= totalCtus) continue;                           // CTA-uniform
    const CtuPos p = ctu_pos(fs, cg);
    ctuX[c] = p.x; ctuY[c] = p.y;
    if (tl) tile_load(tid, fs.rec + (size_t)p.pic * fs.recPicStride, fs.recStride, fs.W, fs.H, p.x, p.y, tl[c]);
  }
  const Row r0 = row_map<LOG2N>(tid, 0);
  const int cg0 = unit * C::CTUS + r0.ctu;
#pragma unroll
  for (int y = 0; y < 8; y++) pre[y] = Vec16{0u, 0u, 0u, 0u};
  if (cg0 < totalCtus) {
    int tx, ty;
    const int16_t* src = frame_src_ptr<LOG2N>(fs, r0, cg0, tx, ty);
    if (tx + 8 <= fs.W && ty + 8 <= fs.H) {
#pragma unroll
      for (int y = 0; y < 8; y++) pre[y] = *reinterpret_cast<const Vec16*>(src + (size_t)y * fs.orgStride);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// border pre-pass of the 8-bit kernel (rmd_border_prep_kernel): one CTA of kTileThreads threads per CTU writes the CTU's images
// (rmd_tc2.cuh PrepSize) of all five depths
// ---------------------------------------------------------------------------------------------
// It stages the reconstruction neighbourhood once (tile_load / tile_store) and then, per depth, runs the prologue's own builders for
// CTU 0 of a CTA of that depth, on a staging area laid out as the RMD CTA's shared memory from VALID_OFF on (rmd_tc2.cuh ProlOff): the PU
// states, the DC sums and the part of the store that CTU 0 touches (N >= 16: both row-group copies, of which the image is the first).
template <int LOG2N>
struct PrepStage {
  typedef tc2::Cfg<LOG2N> C;
  static constexpr int STORE_END = LOG2N == 2 ? 2 * 256 * 16 : (LOG2N == 3 ? 16 : C::GROUP_BYTES + 16) + C::PUS * C::PU_BYTES;
  static constexpr int BYTES = tc2::ProlOff<LOG2N>::STORE + STORE_END;
  static_assert(BYTES % 16 == 0, "the staging is cleared 16 bytes at a time");
};
constexpr int kPrepStageBytes = tc2::cmax(tc2::cmax(tc2::cmax(PrepStage<2>::BYTES, PrepStage<3>::BYTES), tc2::cmax(PrepStage<4>::BYTES, PrepStage<5>::BYTES)),
                                          PrepStage<6>::BYTES);
constexpr int kPrepPhases = 4;      // the kernel syncs its threads after each phase
// Phase `phase` of depth LOG2N for thread tid of CTU cg (origin pos; `tile`: its staged neighbourhood).  img: the pre-pass output,
// kPrepCtuBytes per CTU of the launch.
//   0: clear the staging (so that the bytes no builder writes are the same in every image) and write the PU states of CTU 0; returns
//      whether this thread found a PU to evaluate.  Where no thread did (outside the picture, or pruned in fork-aware mode) the
//      kernel skips phases 1-3: no RMD row consumes that image.
//   1: build_unfiltered   2: build_filtered   3: the image leaves for img
template <int LOG2N>
CUCD_HD int prep_phase(int phase, const FrameSource& fs, int strong, int cg, const CtuPos& pos, const unsigned char* tile, int tid, unsigned char* stage,
                        unsigned char* img) {
  typedef tc2::Cfg<LOG2N> C;
  typedef tc2::PrepSize<LOG2N> S;
  typedef tc2::ProlOff<LOG2N> O;
  constexpr int nthreads = tc2::kTileThreads;
  int any = 0;
  if (phase == 0) {
    Vec16* s = reinterpret_cast<Vec16*>(stage + O::DC);
    for (int i = tid; i < (PrepStage<LOG2N>::BYTES - O::DC) / 16; i += nthreads) s[i] = Vec16{0u, 0u, 0u, 0u};
    const uint8_t* need = ctu_needed<LOG2N>(fs, cg);
    for (int p = tid; p < C::PUS; p += nthreads) {
      stage[p] = pu_state<LOG2N>(fs, need, pos.x, pos.y, p);
      any |= stage[p] == kPuEvaluate;
    }
  } else if (phase == 1) {
    tc2::build_unfiltered_at<LOG2N>(tid, 0, fs.W, fs.H, pos.x, pos.y, tile, stage);
  } else if (phase == 2) {
    tc2::build_filtered_at<LOG2N>(tid, 0, strong, stage);
  } else {
    const Vec16* st = reinterpret_cast<const Vec16*>(stage + O::STORE + tc2::prep_store_off<LOG2N>(0, 0));
    const Vec16* dc = reinterpret_cast<const Vec16*>(stage + O::DC);
    Vec16* d = reinterpret_cast<Vec16*>(img + (size_t)cg * tc2::kPrepCtuBytes + tc2::prep_off<LOG2N>());
    for (int i = tid; i < S::BYTES / 16; i += nthreads) d[i] = i < S::STORE / 16 ? st[i] : dc[i - S::STORE / 16];
  }
  return any;
}

// ---------------------------------------------------------------------------------------------
// copy-out: the cost tables of the unit's CTUs at this depth leave the SM
// ---------------------------------------------------------------------------------------------
// this thread's part of "every PU of the unit's CTUs is evaluated" (the kernel ANDs it over the CTA and with "the unit's last CTU
// exists"): then copy_out skips the state look-up
template <template <int> class Cfg, int LOG2N>
CUCD_HD bool all_evaluated(const uint8_t* valid, int tid, int nthreads) {
  typedef Cfg<LOG2N> C;
  bool mine = true;
  for (int i = tid; i < C::CTUS * 256; i += nthreads) mine = mine && ((i & 255) >= C::PUS || valid[i] == kPuEvaluate);
  return mine;
}
// Element i (= pu * 35 + mode) of CTU c: cost(c, i), the kernel's read-out of its accumulators, for an evaluated PU, the table code
// of a pruned PU or of one outside the picture otherwise.
template <template <int> class Cfg, int LOG2N, class Cost>
CUCD_HD void copy_out(const FrameSource& fs, int unit, int totalCtus, const uint8_t* valid, bool allEval, Cost cost, int tid, int nthreads) {
  typedef Cfg<LOG2N> C;
#pragma unroll 1                                   // unrolled, this loop made ptxas spill in the set-up of tc3_body<5> and <6>
  for (int c = 0; c < C::CTUS; c++) {
    const int cg = unit * C::CTUS + c;
    if (cg >= totalCtus) break;
    const uint8_t* v = valid + c * 256;
    auto val = [&](int i) -> uint32_t {
      const uint8_t s = v[i / kNumModes];
      return s == kPuEvaluate ? cost(c, i) : (s == kPuPruned ? kCostPruned : kCostOutside);
    };
    auto valAll = [&](int i) -> uint32_t { return cost(c, i); };
    if (fs.out) {
      uint32_t* o = fs.out + ((size_t)cg * kPusPerCtu + pu_offset_of_depth(6 - LOG2N)) * kNumModes;
      if (allEval) {
#pragma unroll 4
        for (int i = tid; i < C::PUS * kNumModes; i += nthreads) o[i] = valAll(i);
      } else {
#pragma unroll 4
        for (int i = tid; i < C::PUS * kNumModes; i += nthreads) o[i] = val(i);
      }
    }
    if (fs.outPacked) {
      if (allEval) store_packed_depth<LOG2N>(fs.outPacked + (size_t)cg * kPackedCtuBytes, tid, nthreads, valAll);
      else store_packed_depth<LOG2N>(fs.outPacked + (size_t)cg * kPackedCtuBytes, tid, nthreads, val);
    }
  }
}

}  // namespace tcf
}  // namespace cucd
