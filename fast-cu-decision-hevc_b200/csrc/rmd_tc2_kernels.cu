// rmd_tc2_kernels.cu - tensor-core RMD frame kernel for 8-bit content (sm_100a, tcgen05 kind::i8).
//
// One CTA (256 worker threads = 2 row groups x 128 TMEM lanes, plus one MMA-issuing warp per row group; two CTAs per SM)
// evaluates 2 CTUs (N <= 16) or, in two passes, 4 CTUs (N >= 32) at one depth.  A worker thread owns one 8x8 tile in one
// orientation ("row") for a pass; the issuing warps wait for the rows' arrivals, issue the tcgen05.mma and fetch the
// weights (cp.async.bulk).  Per mode round and row group:
//     gather 32-byte reference window -> shared memory (A1) [N = 4: static 64-byte record row]
//     MMA 1: D1 = A1 x weights(angle, phase)              prediction * 256 in byte 1 of every accumulator
//     epilogue 1: tcgen05.ld.pack::16b + 16 PRMT -> 64 predicted bytes -> TMEM (A2)
//     MMA 2: D2 = source tile (shared memory, static) x -(H8 (x) H8) + A2 x (H8 (x) H8)      Hadamard of the residual
//     epilogue 2: sum |D2|, HM rounding
// See rmd_tc2.cuh for the arithmetic and the reference citations; planar and DC are predicted on the ALU.  The frame-mode set-up
// loads, PU states and copy-out are shared with rmd_tc3_kernels.cu (rmd_tc_frame.cuh), the tcgen05 wrappers live in satd_tc.cuh.
// Replaces, per PU, the reference loop TEncSearch.cpp:2327-2361.
#include <cuda_runtime.h>
#include "rmd_tc2.cuh"
#include "rmd_tc_frame.cuh"
#include "satd_tc.cuh"
#include "kernels.h"

namespace cucd {

extern __shared__ __align__(128) unsigned char smem2[];

using namespace tc;
using namespace tc2;
using namespace tcf;

// CUCD_TC2_TIMING (profiles/ubench/tc2_timing.cu only): per-CTA clock64 stamps of thread 0 at phase boundaries
#ifdef CUCD_TC2_TIMING
__device__ long long* g_tc2Dbg = nullptr;
#ifndef CUCD_TC2_STAMP_TID
#define CUCD_TC2_STAMP_TID 0    // which thread stamps: 0 = the MMA-issuing warp of row group 0, 32 / 96 = other warps of that group
#endif
#define TC2_STAMP(i) do { if (g_tc2Dbg && threadIdx.x == CUCD_TC2_STAMP_TID) g_tc2Dbg[(size_t)blockIdx.x * 64 + (i)] = clock64(); } while (0)
// finer stamps inside the rounds am = 4 (slots 30..) and am = -4 (slots 40..) of the first pass
#define TC2_FINE(i) do { if (g_tc2Dbg && threadIdx.x == CUCD_TC2_STAMP_TID && pass == 0 && (am == 4 || am == -4)) g_tc2Dbg[(size_t)blockIdx.x * 64 + (am == 4 ? 30 : 40) + (i)] = clock64(); } while (0)
#else
#define TC2_STAMP(i) do { } while (0)
#define TC2_FINE(i) do { } while (0)
#endif
// CUCD_TC2_WARPSKEW (profiles/ubench/tc2_skew.cu only): lane 0 of the four warps of row group 0 stamps the events of round am = 4
#ifdef CUCD_TC2_WARPSKEW
__device__ long long* g_tc2Skew = nullptr;
#define TC2_SKEW(e) do { if (g_tc2Skew && pass == 0 && (am == 4 || (am == 3 && (e) < 2)) && (threadIdx.x & 31) == 0 && threadIdx.x < 128) g_tc2Skew[(size_t)blockIdx.x * 64 + (threadIdx.x >> 5) * 16 + (am == 4 ? (e) : 9 + (e))] = clock64(); } while (0)
#else
#define TC2_SKEW(e) do { } while (0)
#endif

namespace {

struct Tc2Args {
  FrameSource fs;             // frame (replay) mode: a unit is a CTU at one depth
  BatchSource bs;             // batch (S2) mode: a unit is 4096 / N^2 caller-described PUs of one size ("virtual CTU")
  int strong, totalCtus;      // totalCtus = number of units
  const uint8_t* tabWin; const uint8_t* tabN4; const int8_t* had;
};

// A CTA = 256 worker threads (the rows) + one MMA-issuing warp per row group.  The workers only ARRIVE on mbarriers when their
// operands are in place; the issuing warp waits for the 128 arrivals, issues the tcgen05.mma and the bulk copy of the next weights
// and commits.  (With the issue inside worker warp 0 that warp ran ~490 cycles behind the other three in every round - the
// tcgen05.wait::st / fence / four UTCIMMA / commit sequence sat on the round's critical path, profiles/ubench/tc2_skew.cu.)
constexpr int kIssuerThreads = 32 * kGroups;
constexpr int kCtaThreads = kThreads + kIssuerThreads;
__device__ __forceinline__ void worker_bar() { asm volatile("bar.sync 1, 256;\n" ::: "memory"); }     // the 256 workers only
// ---- prologue: reference arrays of the CTA's CTUs (rmd_tc2.cuh phases 1-3) --------------------------------
template <int LOG2N, bool FRAME>
__device__ __forceinline__ void tc2_prologue(const Tc2Args& a, const int unit, const TileLoad* tl, const int* ctuX, const int* ctuY) {
  typedef Cfg<LOG2N> C;
  unsigned char* smem = smem2;
  const int tid = threadIdx.x;
  const FrameSource& fs = a.fs;
  if (!FRAME) {
    const BatchSource& bs = a.bs;
    constexpr int TPP = 256 / C::PUS;
#pragma unroll
    for (int c = 0; c < C::CTUS; c++) {
      const int first = (unit * C::CTUS + c) * C::PUS;
      for (int p = tid; p < C::PUS; p += kThreads) smem[C::VALID_OFF + c * 256 + p] = first + p < bs.count ? 1 : 0;
    }
    worker_bar();
#pragma unroll
    for (int c = 0; c < C::CTUS; c++) {
      const int idx = (unit * C::CTUS + c) * C::PUS + tid / TPP;
      build_unfiltered_batch<LOG2N>(tid, c, idx < bs.count ? bs.border + (size_t)bs.pus[idx].borderOff : nullptr, smem);
    }
    if (C::HAS_FILT) {
      worker_bar();
#pragma unroll
      for (int c = 0; c < C::CTUS; c++)
        if ((unit * C::CTUS + c) * C::PUS < bs.count) build_filtered<LOG2N>(tid, c, a.strong, smem);
    }
    return;
  }
#pragma unroll
  for (int c = 0; c < C::CTUS; c++) {
    const int cg = unit * C::CTUS + c;
    uint8_t* valid = smem + C::VALID_OFF + c * 256;
    if (ctuX[c] < 0) {
      for (int p = tid; p < C::PUS; p += kThreads) valid[p] = kPuOutside;
      continue;
    }
    const uint8_t* need = ctu_needed<LOG2N>(fs, cg);
    for (int p = tid; p < C::PUS; p += kThreads) valid[p] = pu_state<LOG2N>(fs, need, ctuX[c], ctuY[c], p);
  }
#pragma unroll
  for (int c = 0; c < C::CTUS; c++)
    if (ctuX[c] >= 0) tile_store<Cfg, LOG2N>(tid, fs.W, fs.H, ctuX[c], ctuY[c], tl[c], smem + C::TILE_OFF + c * C::TILE_BYTES);
  worker_bar();
  TC2_STAMP(51);
#pragma unroll
  for (int c = 0; c < C::CTUS; c++)
    if (ctuX[c] >= 0) build_unfiltered<LOG2N>(tid, c, fs.W, fs.H, ctuX[c], ctuY[c], smem + C::TILE_OFF + c * C::TILE_BYTES, smem);
  TC2_STAMP(52);
  if (C::HAS_FILT) {
    worker_bar();
    TC2_STAMP(53);
#pragma unroll
    for (int c = 0; c < C::CTUS; c++)
      if (ctuX[c] >= 0) build_filtered<LOG2N>(tid, c, a.strong, smem);
  }
}

// ---- the mode rounds of one pass ------------------------------------------------------------------------------
// Per row group the rounds are software pipelined so that the integer ALU has work while an MMA is in flight
// (a lone tcgen05.mma + commit takes ~350 cycles, profiles/ubench):
//     wait MMA1(i) | epilogue 1 -> A2, projected refs of round i+1 | issue MMA2(i) | stage B1/A1 of round i+1 |
//     wait MMA2(i) | issue MMA1(i+1) | epilogue 2 of round i (costs)
// TMEM per row group: D1 = columns [0, 64) (A2 aliases its first 16 once they have been read), D2 = [64, 128).
// `pre`: the eight rows of the source tile of pass 0, loaded by tc2_body before the prologue (frame mode), or nullptr
template <int LOG2N, bool FRAME>
__device__ __forceinline__ void tc2_pass(const Tc2Args& a, const int unit, const int pass, const uint32_t tmemBase, uint32_t& ph1, uint32_t& ph2, const Vec16* pre) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, SEG = RowSeg<LOG2N>::value;
  unsigned char* smem = smem2;
  const int tid = threadIdx.x, grp = tid >> 7, rowTid = tid & 127, warp = tid >> 5, lane = tid & 31;
  const Row r = row_map<LOG2N>(tid, pass);
  unsigned char* store = smem + C::STORE_OFF;
  unsigned char* sA1 = smem + C::A1_OFF + grp * 8192;
  unsigned char* sAorg = smem + C::AORG_OFF + grp * 8192;
  uint64_t* mbar1 = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF) + grp;
  uint64_t* mbar2 = mbar1 + kGroups;
  // "my operands are in place" barriers (128 arrivals each).  Only the issuing warp waits on them: the other three warps of
  // the group arrive and go straight on to their next piece of work instead of idling at a bar.sync.
  uint64_t* arrA = mbar1 + 2 * kGroups;
  uint64_t* arrB = mbar1 + 3 * kGroups;
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  const FrameSource& fs = a.fs;
  const int cg = unit * C::CTUS + r.ctu;
  const bool ok = smem[C::VALID_OFF + r.ctu * 256 + (LOG2N == 2 ? 4 * r.pu : r.pu)] == kPuEvaluate;   // N = 4: the region's PUs share their state (W, H multiples of 8; NxN is pruned as a whole)
  const int slot = pu_slot2<LOG2N>(r.ctu, r.pu);

  uint32_t p[16];                                   // the row's current byte tile: word 2*v + h = pixels (v, 4h..4h+3)
  if (ok) {
    uint32_t raw[16];
    if (FRAME) {
      if (pre && pass == 0) {
#pragma unroll
        for (int y = 0; y < 8; y++) { raw[2 * y] = __byte_perm(pre[y].x, pre[y].y, 0x6420); raw[2 * y + 1] = __byte_perm(pre[y].z, pre[y].w, 0x6420); }
      } else {
        int tx, ty;
        const int16_t* src = frame_src_ptr<LOG2N>(fs, r, cg, tx, ty);
#pragma unroll
        for (int y = 0; y < 8; y++) {
          const uint4 v = *reinterpret_cast<const uint4*>(src + (size_t)y * fs.orgStride);
          raw[2 * y] = __byte_perm(v.x, v.y, 0x6420); raw[2 * y + 1] = __byte_perm(v.z, v.w, 0x6420);
        }
      }
    } else {
      const BatchSource& bs = a.bs;
      const int first = cg * C::PUS;                // cg = index of the virtual CTU
      if (LOG2N == 2) {                             // region = four packed 4x4 blocks (PUs 4*r.pu .. +3, z order: (qy, qx))
#pragma unroll
        for (int q = 0; q < 4; q++) {
          const int idx = first + 4 * r.pu + q;
          uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0;
          if (idx < bs.count) {
            const uint4* b = reinterpret_cast<const uint4*>(bs.org + (size_t)bs.pus[idx].orgOff);
            v0 = b[0]; v1 = b[1];
          }
          // rows of the block: (v0.x, v0.y), (v0.z, v0.w), (v1.x, v1.y), (v1.z, v1.w)
          const int w0 = 2 * ((q >> 1) * 4) + (q & 1);
          raw[w0] = __byte_perm(v0.x, v0.y, 0x6420); raw[w0 + 2] = __byte_perm(v0.z, v0.w, 0x6420);
          raw[w0 + 4] = __byte_perm(v1.x, v1.y, 0x6420); raw[w0 + 6] = __byte_perm(v1.z, v1.w, 0x6420);
        }
      } else {
        const int16_t* src = bs.org + (size_t)bs.pus[first + r.pu].orgOff + (r.o ? r.u0 : r.v0) * N + (r.o ? r.v0 : r.u0);
#pragma unroll
        for (int y = 0; y < 8; y++) {
          const uint4 v = *reinterpret_cast<const uint4*>(src + y * N);
          raw[2 * y] = __byte_perm(v.x, v.y, 0x6420); raw[2 * y + 1] = __byte_perm(v.z, v.w, 0x6420);
        }
      }
    }
    if (r.o) tile_transpose_bytes(raw, p, LOG2N != 2);
    else {
#pragma unroll
      for (int i = 0; i < 16; i++) p[i] = raw[i];
    }
  } else {
#pragma unroll
    for (int i = 0; i < 16; i++) p[i] = 0;
  }

  if (pass == 0) TC2_STAMP(56);
  const uint32_t laneOff = (uint32_t)((warp & 3) * 32) << 16;
  const int rowChunk = (rowTid >> 3) * 128 + (rowTid & 7) * 16;      // the row's 16-byte slot inside a 128-row operand chunk
  const uint32_t tD1 = tmemBase + grp * 128, tA2 = tD1, tD2 = tD1 + 64;
  // the row announces "my A2 is in TMEM" / "my window is in shared memory"; the row group's issuing warp (tc2_issue_pass) does the rest
  auto issue_mma2 = [&]() {
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(arrA);
  };
  auto wait_mma2 = [&]() { mbar_wait(mbar2, ph2); ph2 ^= 1u; tc_fence_after(); };
  auto issue_mma1 = [&]() {
    fence_async_smem();
    tc_fence_before();
    mbar_arrive(arrB);
  };
  auto wait_mma1 = [&]() { mbar_wait(mbar1, ph1); ph1 ^= 1u; tc_fence_after(); };
  // the row's reference window of round `am` into window buffer `buf`
  auto stage_window = [&](int am, int angle, int buf) {
    if (LOG2N == 2) return;
    const int filt = mode_uses_filtered<LOG2N>(26 + am) ? 1 : 0;
    uint32_t w8[8];
    gather_window(store, arr_k0_off<LOG2N>(grp, slot, r.o, filt) + win_k0(angle, r.u0, r.v0), w8);
    uint4* d = reinterpret_cast<uint4*>(sA1 + buf * 4096 + rowChunk);
    d[0] = make_uint4(w8[0], w8[1], w8[2], w8[3]);
    d[128] = make_uint4(w8[4], w8[5], w8[6], w8[7]);          // second 16-byte chunk: + 128 rows * 16 B
  };
  // epilogue 2 + cost hand-over for mode `mode` (has = the row has a mode in this round)
  uint16_t* accN4 = reinterpret_cast<uint16_t*>(acc) + (r.ctu * C::PUS + 4 * r.pu) * kNumModes;
  uint32_t* accRow = acc + (r.ctu * C::PUS + r.pu) * kNumModes;
  auto cost_out = [&](int mode, bool has) {
    // sum |D2| over the row's 64 columns, 16 at a time; the load of chunk c+1 is in flight while chunk c is summed (two independent
    // VABSDIFF chains per chunk), so one TMEM load latency is exposed per epilogue instead of one per load
    uint32_t q[4];
    uint32_t va[16], vb[16];
    auto sum16 = [](const uint32_t* v) {
      uint32_t s0 = 0, s1 = 0;
#pragma unroll
      for (int k = 0; k < 8; k++) { s0 = sad_acc(v[k], 0u, s0); s1 = sad_acc(v[8 + k], 0u, s1); }
      return s0 + s1;
    };
    tmem_ld16(tD2 + laneOff, va);
    tmem_ld_wait();
    tmem_ld16(tD2 + laneOff + 16, vb);
    q[0] = sum16(va);
    tmem_ld_wait();
    tmem_ld16(tD2 + laneOff + 32, va);
    q[1] = sum16(vb);
    tmem_ld_wait();
    tmem_ld16(tD2 + laneOff + 48, vb);
    q[2] = sum16(va);
    tmem_ld_wait();
    q[3] = sum16(vb);
    tc_fence_before();
    if (LOG2N == 2) {
      if (ok && has) {
#pragma unroll
        for (int c = 0; c < 4; c++) accN4[c * kNumModes + mode] = (uint16_t)((q[c] + 1u) >> 1);   // xCalcHADs4x4 rounding; 8-bit: no final shift
      }
    } else {
      uint32_t v = ok ? ((q[0] + q[1] + q[2] + q[3] + 2u) >> 2) : 0u;                    // xCalcHADs8x8 rounding
#pragma unroll
      for (int m = 1; m < SEG; m <<= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
      if (ok && has && (lane & (SEG - 1)) == 0) {
        if (LOG2N >= 4) atomicAdd(accRow + mode, v); else accRow[mode] = v;
      }
    }
  };

  // ---- the row's source tile becomes the static A operand of the -H product -------------------------------------
  {
    uint4* d = reinterpret_cast<uint4*>(sAorg + rowChunk);
#pragma unroll
    for (int i = 0; i < 4; i++) d[i * 128] = make_uint4(p[4 * i], p[4 * i + 1], p[4 * i + 2], p[4 * i + 3]);
  }
  const unsigned char* rec4 = store + rec_off(r.ctu, r.o, 4 * r.pu);
  if (LOG2N == 2) {                                 // N = 4: the record row is the A operand of every mode (4 chunks)
    uint4* d = reinterpret_cast<uint4*>(sA1 + rowChunk);
#pragma unroll
    for (int i = 0; i < 4; i++) d[i * 128] = reinterpret_cast<const uint4*>(rec4)[i];
  }
  // round 0 prediction: planar (true orientation rows) / DC (transposed rows) on the ALU
  const unsigned char* unfMain = store + arr_k0_off<LOG2N>(grp, slot, r.o, 0);
  const unsigned char* unfSide = store + arr_k0_off<LOG2N>(grp, slot, r.o ^ 1, 0);
  if (ok) {
    if (LOG2N == 2) { if (r.o == 0) planar_region4(rec4, p); else dc_region4(rec4, p); }
    else if (r.o == 0) {
      constexpr int f = C::HAS_FILT ? 1 : 0;        // planar reads the smoothed border for N = 8, 16, 32 (TComPattern.cpp:523-548)
      planar_tile(LOG2N, store + arr_k0_off<LOG2N>(grp, slot, 0, f), store + arr_k0_off<LOG2N>(grp, slot, 1, f), r.u0, r.v0, p);
    } else {
      dc_tile((reinterpret_cast<const int*>(smem + C::DC_OFF)[r.ctu * 64 + r.pu] + N) >> (LOG2N + 1), C::EDGE, unfMain, unfSide, r.u0, r.v0, p);
    }
  }
  fence_async_smem();                               // the source operand is read by the tensor core (async proxy)
  if (pass == 0) TC2_STAMP(57);

  // ---- round 0 -------------------------------------------------------------------------------------------------
  tmem_st16(tA2 + laneOff, p);
  issue_mma2();
  stage_window(8, 32, 0);
  wait_mma2();
  issue_mma1();
  cost_out(r.o ? 1 : 0, true);
  if (pass == 0) TC2_STAMP(8);

  // ---- angular rounds -----------------------------------------------------------------------------------------
  int angle = 32, angleNext = 26;
#pragma unroll 1
  for (int am = 8; am >= -8; --am) {
    const int buf = (8 - am) & 1;
    const int angleNext2 = am > -7 ? angle_of_am(am - 2) : 0;
    TC2_FINE(0);
    TC2_SKEW(0);
    wait_mma1();
    TC2_FINE(1);
    TC2_SKEW(1);
    // epilogue 1: byte 1 of every accumulator is the predicted pixel
    {
      uint32_t v[32];
      tmem_ld16_pack(tD1 + laneOff, v);
      tmem_ld16_pack(tD1 + laneOff + 32, v + 16);
      tmem_ld_wait();
      pack_pred(v, p, 8);
      pack_pred(v + 16, p + 8, 8);
    }
    if (C::EDGE && am == 0 && ok) {
      if (LOG2N == 2) patch_edge0_region4(rec4, p);
      else if (r.u0 == 0) patch_edge0_tile(unfMain, unfSide, r.v0, p);
    }
    tmem_st16(tA2 + laneOff, p);
    TC2_FINE(2);
    TC2_SKEW(2);
    // Projected samples of the next (negative) angle.  The gathers of round am have all finished: MMA 1 of this round was only
    // issued after every row of the group had announced its window (arrB).  The OTHER rows' projected samples are complete once
    // MMA 2 below has been issued (every row announces arrA after this point), i.e. after wait_mma2: a window that may read
    // them is gathered there, one that cannot (angle >= 0) right away, under the MMA.
    const bool lateWindow = LOG2N != 2 && am > -8 && angleNext < 0;
    if (lateWindow) build_ext_group<LOG2N>(rowTid, grp, inv_angle_of_am(am - 1), mode_uses_filtered<LOG2N>(25 + am) ? 1 : 0, store);
    TC2_FINE(3);
    TC2_SKEW(3);
    issue_mma2();
    TC2_FINE(4);
    TC2_SKEW(4);
    if (am > -8) {
      if (!lateWindow) stage_window(am - 1, angleNext, buf ^ 1);
    }
    TC2_FINE(5);
    TC2_SKEW(5);
    wait_mma2();
    TC2_FINE(6);
    TC2_SKEW(6);
    if (lateWindow) stage_window(am - 1, angleNext, buf ^ 1);
    if (am > -8) issue_mma1();
    TC2_FINE(7);
    TC2_SKEW(7);
    cost_out(r.o ? 10 - am : 26 + am, !(r.o && am == -8));
    TC2_FINE(8);
    TC2_SKEW(8);
    if (pass == 0) TC2_STAMP(9 + 8 - am);
    angle = angleNext; angleNext = angleNext2;
  }
  (void)angle;
}

// ---- the MMA-issuing warp of row group `g` (threads 256 + 32 g ...): one pass ---------------------------------------------
// Mirrors the workers' sequence of tc2_pass: round 0 (MMA 2 only), then per angular round MMA 2 of the round and MMA 1 of the next.
// The weights of round am - 2 are fetched (cp.async.bulk, completion on barT) right after MMA 1 of round am - 1 has been issued,
// into the buffer MMA 1 of round am has finished with (the workers passed wait_mma1 of that round before they arrived here).
template <int LOG2N>
__device__ __forceinline__ void tc2_issue_pass(const Tc2Args& a, const int pass, const uint32_t tmemBase, const int g, uint32_t& phA, uint32_t& phB, uint32_t& phT) {
  typedef Cfg<LOG2N> C;
  unsigned char* smem = smem2;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint64_t* bar1 = bars + g;
  uint64_t* bar2 = bars + kGroups + g;
  uint64_t* arrA = bars + 2 * kGroups + g;
  uint64_t* arrB = bars + 3 * kGroups + g;
  uint64_t* barT = bars + 4 * kGroups + g;
  const uint32_t uD1 = tmemBase + g * 128, uA2 = uD1, uD2 = uD1 + 64;
  unsigned char* sB1 = smem + C::B1_OFF + g * 2 * C::B1_BYTES;
  const uint32_t idescPred = make_idesc_i8(128, 64, 0, 0), idescHad = make_idesc_i8(128, 64, 0, 1);
  const uint64_t dHad = make_desc(smem_u32(smem + C::HAD_OFF), 1024, 128), dHadNeg = make_desc(smem_u32(smem + C::HAD_OFF + 4096), 1024, 128);
  const uint64_t dAorg = make_desc(smem_u32(smem + C::AORG_OFF + g * 8192), 2048, 128);
  const uint64_t dB1 = make_desc(smem_u32(sB1), 1024, 128), dA1 = make_desc(smem_u32(smem + C::A1_OFF + g * 8192), 2048, 128);
  constexpr uint64_t kStepB = (2 * 1024) >> 4;      // descriptor advance of one K = 32 step: two 16-byte chunks of 64 rows
  constexpr uint64_t kStepA = (2 * 2048) >> 4;      // ... of 128 rows
  const bool lead = elect_one();

  auto fetch = [&](int am, int buf) {               // weights of round `am` -> buffer `buf`
    if (lead) {
      const int ai = am + 8;
      const uint8_t* src = LOG2N == 2 ? a.tabN4 + ai * 4096 : a.tabWin + (ai * 4 + (group_frac0<LOG2N>(g, pass, angle_of_am(am)) >> 3)) * 2048;
      mbar_expect_tx(barT, C::B1_BYTES);
      bulk_g2s(sB1 + buf * C::B1_BYTES, src, C::B1_BYTES, barT);
    }
  };
  // source x -H + A2 (stored to TMEM by every row) x H -> D2
  auto mma2 = [&]() {
    mbar_wait(arrA, phA); phA ^= 1u;
    tc_fence_after();
    if (lead) {
      mma_i8(uD2, dAorg, dHadNeg, idescHad, 0u);
      mma_i8(uD2, dAorg + kStepA, dHadNeg + kStepB, idescHad, 1u);
      mma_i8_ts(uD2, uA2, dHad, idescHad, 1u);
      mma_i8_ts(uD2, uA2 + 8, dHad + kStepB, idescHad, 1u);
      mma_commit(bar2);
    }
    __syncwarp();
  };
  // window / record operand (shared memory) x weights -> D1
  auto mma1 = [&](int buf) {
    mbar_wait(arrB, phB); phB ^= 1u;
    mbar_wait(barT, phT); phT ^= 1u;
    tc_fence_after();
    if (lead) {
      const uint64_t dB = dB1 + (uint64_t)((buf * C::B1_BYTES) >> 4);
      if (LOG2N == 2) {
        mma_i8(uD1, dA1, dB, idescPred, 0u);
        mma_i8(uD1, dA1 + kStepA, dB + kStepB, idescPred, 1u);
      } else {
        mma_i8(uD1, dA1 + (uint64_t)((buf * 4096) >> 4), dB, idescPred, 0u);
      }
      mma_commit(bar1);
    }
    __syncwarp();
  };
  fetch(8, 0);
  mma2();                                           // round 0: planar / DC
  mma1(0);
  fetch(7, 1);
#pragma unroll 1
  for (int am = 8; am >= -8; --am) {
    const int buf = (8 - am) & 1;
    mma2();
    if (am > -8) {
      mma1(buf ^ 1);
      if (am > -7) fetch(am - 2, buf);
    }
  }
}

template <int LOG2N, bool FRAME>
__device__ __noinline__ void tc2_body(const Tc2Args& a, const int unit) {
  typedef Cfg<LOG2N> C;
  unsigned char* smem = smem2;
  const int tid = threadIdx.x, warp = tid >> 5;
  const bool worker = tid < kThreads;               // threads 256.. are the MMA-issuing warps (tc2_issue_pass)
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  if (FRAME && a.fs.needed) {
    // fork-aware mode: a CTA none of whose PUs has to be evaluated writes the table codes and leaves
    const int any = worker ? fork_states<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, tid, kThreads) : 0;
    if (!__syncthreads_or(any)) {
      if (worker) copy_out<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, false, CostRead<LOG2N>{acc}, tid, kThreads);
      return;
    }
    if (worker) worker_bar();
  }
  uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(smem + C::BAR_OFF + 96);
  if (tid == 0) {
    for (int i = 0; i < 5 * kGroups; i++)           // MMA done x2 (1 arrival: the commit), operands ready x2 (128 rows), weights landed (1 + bytes)
      mbar_init(reinterpret_cast<uint64_t*>(smem + C::BAR_OFF) + i, (i >= 2 * kGroups && i < 4 * kGroups) ? 128 : 1);
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  uint32_t ph1 = 0, ph2 = 0;
  Vec16 pre[8];
  if (worker) {
  TC2_STAMP(0);
  if (warp == 0) tmem_alloc(tmemSlot, 256);
  TC2_STAMP(58);
  // Every global load of the set-up is issued here, before anything waits: the Hadamard operands, the reconstruction
  // neighbourhoods of the CTA's CTUs (tile_load) and the rows' source tiles of pass 0 share ONE memory round trip.
  const uint4 hadP = reinterpret_cast<const uint4*>(a.had + (LOG2N == 2 ? 8192 : 0))[tid];        // +H
  const uint4 hadN = reinterpret_cast<const uint4*>(a.had + (LOG2N == 2 ? 8192 : 0))[tid + 256];  // -H
  int ctuX[C::CTUS], ctuY[C::CTUS];
  TileLoad tl[C::CTUS];
  if (FRAME) setup_loads<Cfg, LOG2N>(a.fs, unit, a.totalCtus, tid, ctuX, ctuY, tl, pre);
  TC2_STAMP(59);
  if (LOG2N >= 4) for (int i = tid; i < C::CTUS * C::PUS * kNumModes; i += kThreads) acc[i] = 0;   // accumulated with atomics
  reinterpret_cast<int*>(smem + C::DC_OFF)[tid] = 0;          // CTUS * 64 <= 256 sums
  reinterpret_cast<uint4*>(smem + C::HAD_OFF)[tid] = hadP;
  TC2_STAMP(60);
  reinterpret_cast<uint4*>(smem + C::HAD_OFF)[tid + 256] = hadN;
  worker_bar();
  TC2_STAMP(50);
  tc2_prologue<LOG2N, FRAME>(a, unit, tl, ctuX, ctuY);
  TC2_STAMP(54);
  tc_fence_before();
  fence_async_smem();
  }                                                 // if (worker)
  __syncthreads();                                  // barriers initialised, TMEM allocated, operands of the set-up visible: workers and issuers
  tc_fence_after();
  const uint32_t tmemBase = *tmemSlot;
  TC2_STAMP(1);
  if (worker) {
#pragma unroll 1
    for (int pass = 0; pass < C::PASSES; pass++) tc2_pass<LOG2N, FRAME>(a, unit, pass, tmemBase, ph1, ph2, FRAME ? pre : nullptr);
  } else {
    uint32_t phA = 0, phB = 0, phT = 0;
#pragma unroll 1
    for (int pass = 0; pass < C::PASSES; pass++) tc2_issue_pass<LOG2N>(a, pass, tmemBase, warp - kThreads / 32, phA, phB, phT);
  }
  TC2_STAMP(2);

  // ---- costs leave the SM ------------------------------------------------------------------------------------
  tc_fence_before();
  // the common case - every PU of the CTA evaluated - copies the accumulators without a per-element state look-up
  bool mine = true;
  if (FRAME && worker) mine = all_evaluated<Cfg, LOG2N>(smem + C::VALID_OFF, tid, kThreads);
  const bool allEval = __syncthreads_and(mine) && unit * C::CTUS + C::CTUS <= a.totalCtus;
  if (!worker) return;
  if (!FRAME) {
    // batch mode: row outIndex of the caller's [nPU][35] table per PU
    const BatchSource& bs = a.bs;
    for (int i = tid; i < C::CTUS * C::PUS * kNumModes; i += kThreads) {
      const int pl = i / kNumModes, m = i - pl * kNumModes, idx = unit * C::CTUS * C::PUS + pl;
      if (idx >= bs.count) continue;
      bs.out[(size_t)bs.pus[idx].outIndex * kNumModes + m] = CostRead<LOG2N>{acc}(0, i);
    }
    if (warp == 0) tmem_dealloc(tmemBase, 256);
    return;
  }
  copy_out<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, allEval, CostRead<LOG2N>{acc}, tid, kThreads);
  if (warp == 0) tmem_dealloc(tmemBase, 256);
  TC2_STAMP(3);
#ifdef CUCD_TC2_TIMING
  if (g_tc2Dbg && tid == 0) g_tc2Dbg[(size_t)blockIdx.x * 64 + 4] = LOG2N;
#endif
}

// blocks of one launch: depth-major (rmd_tc_frame.cuh frame_block)
__global__ void __launch_bounds__(kCtaThreads, 2)
rmd_frame_tc2_kernel(const __grid_constant__ Tc2Args a) {
  const FrameBlock fb = frame_block(a.totalCtus, blockIdx.x);
  switch (fb.log2n) {
    case 6: tc2_body<6, true>(a, fb.unit); break;
    case 5: tc2_body<5, true>(a, fb.unit); break;
    case 4: tc2_body<4, true>(a, fb.unit); break;
    case 3: tc2_body<3, true>(a, fb.unit); break;
    default: tc2_body<2, true>(a, fb.unit);
  }
}

// batch (S2) mode: one launch per PU size
template <int LOG2N>
__global__ void __launch_bounds__(kCtaThreads, 2)
rmd_batch_tc2_kernel(const __grid_constant__ Tc2Args a) { tc2_body<LOG2N, false>(a, blockIdx.x); }

template <int LOG2N>
cudaError_t launch_batch_tc2(const Tc2Args& a, int units, cudaStream_t st) {
  rmd_batch_tc2_kernel<LOG2N><<<(units + Cfg<LOG2N>::CTUS - 1) / Cfg<LOG2N>::CTUS, kCtaThreads, Cfg<LOG2N>::TOTAL, st>>>(a);
  return cudaGetLastError();
}

}  // namespace

int rmd_tc2_smem_bytes() { return kSmemBytes; }

// per-device opt-in to > 48 KB of dynamic shared memory (called by cucd_create after cudaSetDevice)
cudaError_t configure_rmd_tc2_kernels() {
  cudaError_t e = cudaFuncSetAttribute(rmd_frame_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(rmd_batch_tc2_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<2>::TOTAL);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(rmd_batch_tc2_kernel<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<3>::TOTAL);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(rmd_batch_tc2_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<4>::TOTAL);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(rmd_batch_tc2_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<5>::TOTAL);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(rmd_batch_tc2_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<6>::TOTAL);
  return e;
}

cudaError_t launch_rmd_batch_tc2(int log2n, const BatchSource& bs, int strong, const uint8_t* tabWin, const uint8_t* tabN4, const int8_t* hadamard,
                                 cudaStream_t st, int* launches) {
  if (bs.count <= 0) return cudaSuccess;
  const int n = 1 << log2n, pus = 4096 / (n * n);
  Tc2Args a;
  a.fs = FrameSource{}; a.bs = bs; a.strong = strong; a.totalCtus = (bs.count + pus - 1) / pus; a.tabWin = tabWin; a.tabN4 = tabN4; a.had = hadamard;
  cudaError_t e;
  switch (log2n) {
    case 2: e = launch_batch_tc2<2>(a, a.totalCtus, st); break;
    case 3: e = launch_batch_tc2<3>(a, a.totalCtus, st); break;
    case 4: e = launch_batch_tc2<4>(a, a.totalCtus, st); break;
    case 5: e = launch_batch_tc2<5>(a, a.totalCtus, st); break;
    case 6: e = launch_batch_tc2<6>(a, a.totalCtus, st); break;
    default: return cudaErrorInvalidValue;
  }
  if (e == cudaSuccess && launches) *launches += 1;
  return e;
}

cudaError_t launch_rmd_frames_tc2(const FrameSource& fs, int nPics, int strong, const uint8_t* tabWin, const uint8_t* tabN4, const int8_t* hadamard,
                                  cudaStream_t st, int* launches) {
  const int total = nPics * fs.ctusPerPic;
  if (total <= 0) return cudaSuccess;
  Tc2Args a;
  a.fs = fs; a.bs = BatchSource{}; a.strong = strong; a.totalCtus = total; a.tabWin = tabWin; a.tabN4 = tabN4; a.had = hadamard;
  rmd_frame_tc2_kernel<<<frame_blocks(total), kCtaThreads, kSmemBytes, st>>>(a);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace cucd
