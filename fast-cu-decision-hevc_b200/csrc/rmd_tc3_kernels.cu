// rmd_tc3_kernels.cu - tensor-core RMD frame kernel for 9/10-bit content (sm_100a, tcgen05 kind::f16, fp32 accumulators).
//
// The work decomposition, row map and software pipeline are those of rmd_tc2_kernels.cu (256 threads = 2 row groups x 128
// TMEM lanes, two CTAs per SM, a thread owns one 8x8 tile in one orientation for a pass); the operands are half precision
// holding exact integers (rmd_tc3.cuh).  Per mode round and row group:
//     gather 24 reference samples (fp16 1024 + s) -> shared memory (A1)      [N = 4: static records, written by the prologue]
//     MMA 1: D1 = A1 x weights(angle, phase) = 2^23 + 32768 + 32 * pred + remainder      (weights arrive by cp.async.bulk)
//     epilogue 1: tcgen05.ld.pack::16b, (x >> 5) & 0x3ff | 0x6400 -> 64 predicted fp16 (1024 + pred)
//     (epilogue 1 also subtracts the row's source tile: A2 = pred - src, exact in fp16)
//     MMA 2: D2 = A2 x H                                                                   Hadamard of the residual
//     epilogue 2: sum |D2| with FADD |x| (exact), HM rounding, >> (bitDepth - 8)
// Differences that matter: single-buffered operands (MMA 1 of a round has completed before the next round is staged), the
// MMA 1 weights are fetched by one elected lane with a bulk copy that completes on an mbarrier (no registers, no LDG/STS per
// thread), N = 4 runs four N = 16, K = 16 products per MMA against one 512-byte table, and every operand byte the tensor
// core can see is a finite number (the stores are zeroed first: 0 x NaN would poison an accumulator).
// The frame-mode set-up loads, PU states and copy-out are those of rmd_tc2_kernels.cu (rmd_tc_frame.cuh), the tcgen05 wrappers
// live in satd_tc.cuh.
// Replaces, per PU, the reference loop TEncSearch.cpp:2327-2361 for internal bit depths 9 and 10 (8 also works and is tested).
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include "rmd_tc3.cuh"
#include "rmd_tc_frame.cuh"
#include "satd_tc.cuh"
#include "kernels.h"

namespace cucd {

extern __shared__ __align__(128) unsigned char smem3[];

using namespace tc;
using namespace tc3;
using namespace tcf;

namespace {

struct Tc3Args {
  FrameSource fs;
  int strong, totalCtus, bitDepth;
  const uint8_t* tabWin; const uint8_t* tabN4; const uint8_t* had;
};

// ---- prologue: reference arrays of the CTA's CTUs (rmd_tc3.cuh phases 1-3) --------------------------------
template <int LOG2N>
__device__ __forceinline__ void tc3_prologue(const Tc3Args& a, const int unit, const TileLoad* tl, const int* ctuX, const int* ctuY) {
  typedef Cfg<LOG2N> C;
  unsigned char* smem = smem3;
  const int tid = threadIdx.x;
  const FrameSource& fs = a.fs;
#pragma unroll
  for (int c = 0; c < C::CTUS; c++) {
    const int cg = unit * C::CTUS + c;
    uint8_t* valid = smem + C::VALID_OFF + c * 256;
    if (ctuX[c] < 0) {                                         // CTA-uniform
      for (int p = tid; p < C::PUS; p += kThreads) valid[p] = kPuOutside;
      continue;
    }
    const uint8_t* need = ctu_needed<LOG2N>(fs, cg);
    for (int p = tid; p < C::PUS; p += kThreads) valid[p] = pu_state<LOG2N>(fs, need, ctuX[c], ctuY[c], p);
    tile_store<Cfg, LOG2N>(tid, fs.W, fs.H, ctuX[c], ctuY[c], tl[c], reinterpret_cast<uint16_t*>(smem + C::TILE_OFF + c * C::TILE_BYTES));
  }
  __syncthreads();
#pragma unroll
  for (int c = 0; c < C::CTUS; c++)
    if (ctuX[c] >= 0)
      build_unfiltered16<LOG2N>(tid, c, fs.W, fs.H, ctuX[c], ctuY[c], a.bitDepth, reinterpret_cast<const uint16_t*>(smem + C::TILE_OFF + c * C::TILE_BYTES), smem);
  if (C::HAS_FILT) {
    __syncthreads();
#pragma unroll
    for (int c = 0; c < C::CTUS; c++)
      if (ctuX[c] >= 0) build_filtered16<LOG2N>(tid, c, a.strong, a.bitDepth, smem);
  }
}

// ---- the mode rounds of one pass (pipeline of rmd_tc2_kernels.cu tc2_pass) ------------------------------------------
// TMEM per row group: D1 = columns [0, 64) (A2 aliases its first 32 once they have been read), D2 = [64, 128).
// `pre`: the eight rows of the source tile of pass 0, loaded by tc3_body before the prologue
template <int LOG2N>
__device__ __forceinline__ void tc3_pass(const Tc3Args& a, const int unit, const int pass, const uint32_t tmemBase, uint32_t& ph1, uint32_t& ph2,
                                         uint32_t& phA, uint32_t& phB, uint32_t& phT, const Vec16* pre) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, SEG = RowSeg<LOG2N>::value;
  unsigned char* smem = smem3;
  const int tid = threadIdx.x, grp = tid >> 7, rowTid = tid & 127, warp = tid >> 5, lane = tid & 31;
  const Row r = row_map<LOG2N>(tid, pass);
  unsigned char* store = smem + C::STORE_OFF;
  unsigned char* sA1 = smem + C::A1_OFF + grp * C::A1_BYTES;
  unsigned char* sAorg = smem + C::AORG_OFF + grp * C::AORG_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint64_t* mbar1 = bars + grp;                   // MMA 1 done
  uint64_t* mbar2 = bars + kGroups + grp;         // MMA 2 done
  uint64_t* arrA = bars + 2 * kGroups + grp;      // "my A2 is in TMEM" (128 arrivals, only the issuing warp waits)
  uint64_t* arrB = bars + 3 * kGroups + grp;      // "my window is in shared memory"
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  const FrameSource& fs = a.fs;
  const int cg = unit * C::CTUS + r.ctu;
  const bool ok = smem[C::VALID_OFF + r.ctu * 256 + (LOG2N == 2 ? 4 * r.pu : r.pu)] == kPuEvaluate;
  const int slot = pu_slot<LOG2N>(r.ctu, r.pu);
  const int maxVal = (1 << a.bitDepth) - 1, shift = a.bitDepth - 8;
  const int rowChunk = row_chunk(rowTid);

  uint32_t p[32];                                   // the row's current tile as fp16 pairs: word = pixels (2w, 2w + 1)
  if (ok) {
    uint32_t raw[32];
    if (pass == 0) {
#pragma unroll
      for (int y = 0; y < 8; y++) { raw[4 * y] = pre[y].x; raw[4 * y + 1] = pre[y].y; raw[4 * y + 2] = pre[y].z; raw[4 * y + 3] = pre[y].w; }
    } else {
      int tx, ty;
      const int16_t* src = frame_src_ptr<LOG2N>(fs, r, cg, tx, ty);
#pragma unroll
      for (int y = 0; y < 8; y++) {
        const uint4 v = *reinterpret_cast<const uint4*>(src + (size_t)y * fs.orgStride);
        raw[4 * y] = v.x; raw[4 * y + 1] = v.y; raw[4 * y + 2] = v.z; raw[4 * y + 3] = v.w;
      }
    }
    if (LOG2N == 2) region_to_quadrants16(raw, p, r.o != 0);
    else if (r.o) tile_transpose16(raw, p);
    else {
#pragma unroll
      for (int i = 0; i < 32; i++) p[i] = raw[i];
    }
#pragma unroll
    for (int i = 0; i < 32; i++) p[i] = (p[i] & kMask2) | kBias2;
  } else {
#pragma unroll
    for (int i = 0; i < 32; i++) p[i] = 0;
  }

  const uint32_t laneOff = (uint32_t)((warp & 3) * 32) << 16;
  const uint32_t tD1 = tmemBase + grp * 128, tA2 = tD1, tD2 = tD1 + 64;
  // what the MMA-issuing lane needs, from warp-uniform values (see rmd_tc2_kernels.cu)
  const int warpU = __shfl_sync(0xffffffffu, warp, 0), grpU = warpU >> 2;
  const bool issuer = (warpU & 3) == 0;
  const uint32_t tmemU = __shfl_sync(0xffffffffu, tmemBase, 0);
  const uint32_t uD1 = tmemU + grpU * 128, uA2 = uD1, uD2 = uD1 + 64;
  uint64_t* ubar1 = bars + grpU;
  uint64_t* ubar2 = bars + kGroups + grpU;
  uint64_t* uarrA = bars + 2 * kGroups + grpU;
  uint64_t* uarrB = bars + 3 * kGroups + grpU;
  uint64_t* ubarT = bars + 4 * kGroups + grpU;    // weights of the next MMA 1 have landed
  unsigned char* uB1 = smem + C::B1_OFF + grpU * C::B1_BYTES;
  constexpr int NB = LOG2N == 2 ? 16 : 64;          // N of one MMA (N = 4: one quadrant)
  constexpr uint32_t kLboB = NB * 16;               // bytes between 16-byte K chunks of a B operand
  const uint32_t idescPred = make_idesc_f16(128, NB, 0), idescHad = make_idesc_f16(128, NB, 0);
  const uint64_t dHad = make_desc(smem_u32(smem + C::HAD_OFF), kLboB, 128);
  const uint64_t dB1 = make_desc(smem_u32(uB1), kLboB, 128), dA1 = make_desc(smem_u32(smem + C::A1_OFF + grpU * C::A1_BYTES), 2048, 128);
  constexpr uint64_t kStepB = (2 * kLboB) >> 4;     // descriptor advance of one K = 16 step: two 16-byte chunks
  constexpr uint64_t kStepA = (2 * 2048) >> 4;      // ... of 128 rows

  // -(source) x H + A2 (already stored to TMEM by every thread) x H -> D2
  auto arrive_mma2 = [&]() {
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(arrA);
  };
  auto fire_mma2 = [&]() {
    if (issuer) {
      mbar_wait(uarrA, phA);
      tc_fence_after();
      if (elect_one()) {
        // A2 holds the residual pred - src itself (exact in fp16: |.| <= 1023): one product, no source operand
        if (LOG2N == 2) {
#pragma unroll
          for (int q = 0; q < 4; q++) mma_f16_ts(uD2 + 16 * q, uA2 + 8 * q, dHad, idescHad, 0u);
        } else {
#pragma unroll
          for (int s = 0; s < 4; s++) mma_f16_ts(uD2, uA2 + 8 * s, dHad + s * kStepB, idescHad, s ? 1u : 0u);
        }
        mma_commit(ubar2);
      }
      __syncwarp();
    }
    phA ^= 1u;
  };
  auto issue_mma2 = [&]() { arrive_mma2(); fire_mma2(); };
  auto wait_mma2 = [&]() { mbar_wait(mbar2, ph2); ph2 ^= 1u; tc_fence_after(); };
  // window / record operand (shared memory) x weights -> D1
  auto issue_mma1 = [&]() {
    fence_async_smem();
    tc_fence_before();
    mbar_arrive(arrB);
    if (issuer) {
      mbar_wait(uarrB, phB);
      mbar_wait(ubarT, phT);
      tc_fence_after();
      if (elect_one()) {
        if (LOG2N == 2) {
#pragma unroll
          for (int q = 0; q < 4; q++) mma_f16_ss(uD1 + 16 * q, dA1 + q * kStepA, dB1, idescPred, 0u);
        } else {
          mma_f16_ss(uD1, dA1, dB1, idescPred, 0u);
          mma_f16_ss(uD1, dA1 + kStepA, dB1 + kStepB, idescPred, 1u);
        }
        mma_commit(ubar1);
      }
      __syncwarp();
    }
    phB ^= 1u; phT ^= 1u;
  };
  auto wait_mma1 = [&]() { mbar_wait(mbar1, ph1); ph1 ^= 1u; tc_fence_after(); };
  // weights of round `am`: one bulk copy per row group.  The buffer is free: the MMA 1 that read it has completed.
  auto fetch_weights = [&](int am, int angle) {
    if (issuer) {
      if (elect_one()) {
        const uint8_t* src = LOG2N == 2 ? a.tabN4 + (am + 8) * kN4Table16
                                        : a.tabWin + ((am + 8) * 4 + (group_frac0<LOG2N>(grpU, pass, angle) >> 3)) * kWinTable16;
        mbar_expect_tx(ubarT, C::B1_BYTES);
        bulk_g2s(uB1, src, C::B1_BYTES, ubarT);
      }
      __syncwarp();
    }
  };
  auto stage_window = [&](int am, int angle) {
    if (LOG2N == 2) return;
    const int filt = mode_uses_filtered<LOG2N>(26 + am) ? 1 : 0;
    uint32_t w[12];
    gather_window16(store, arr_k0_off<LOG2N>(grp, slot, r.o, filt) + 2 * win_k0(angle, r.u0, r.v0), w);
    uint4* d = reinterpret_cast<uint4*>(sA1 + rowChunk);
    d[0] = make_uint4(w[0], w[1], w[2], w[3]);
    d[128] = make_uint4(w[4], w[5], w[6], w[7]);            // next 16-byte chunk: + 128 rows * 16 B
    d[256] = make_uint4(w[8], w[9], w[10], w[11]);
  };
  // A2 = (1024 + pred) - (1024 + src) per half = the residual itself, exact in fp16 (|pred - src| <= 1023): MMA 2 needs no source
  // operand.  The row reads its source tile back from its own slot of the source buffer (written once per pass, below).
  auto store_a2 = [&](uint32_t* q) {
    const uint4* sv = reinterpret_cast<const uint4*>(sAorg + rowChunk);
    auto sub2 = [](uint32_t x, uint32_t y) {
      const __half2 d = __hsub2(*reinterpret_cast<const __half2*>(&x), *reinterpret_cast<const __half2*>(&y));
      return *reinterpret_cast<const uint32_t*>(&d);
    };
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const uint4 o = sv[i * 128];
      q[4 * i] = sub2(q[4 * i], o.x); q[4 * i + 1] = sub2(q[4 * i + 1], o.y); q[4 * i + 2] = sub2(q[4 * i + 2], o.z); q[4 * i + 3] = sub2(q[4 * i + 3], o.w);
    }
    tmem_st32(tA2 + laneOff, q);
  };
  auto rec = [&](int q, int s) { return ld_s16(smem + rec_slot_off(r.ctu, r.o, 4 * r.pu + q, s)); };
  // epilogue 2 + cost hand-over for mode `mode` (has = the row has a mode in this round)
  uint16_t* acc16 = reinterpret_cast<uint16_t*>(acc);
  auto cost_out = [&](int mode, bool has) {
    float q[4];
    uint32_t va[16], vb[16];
    auto sum16 = [](const uint32_t* v) {
      float s0 = 0.f, s1 = 0.f;
#pragma unroll
      for (int k = 0; k < 8; k++) { s0 += fabsf(__uint_as_float(v[k])); s1 += fabsf(__uint_as_float(v[8 + k])); }
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
        for (int c = 0; c < 4; c++)        // xCalcHADs4x4 rounding, then xGetHADs' precision adjustment (TComRdCost.cpp:1343-1411, 1603)
          acc16[(r.ctu * C::PUS + 4 * r.pu + c) * kNumModes + mode] = (uint16_t)(((__float2uint_rz(q[c]) + 1u) >> 1) >> shift);
      }
    } else {
      uint32_t v = ok ? ((__float2uint_rz((q[0] + q[1]) + (q[2] + q[3])) + 2u) >> 2) : 0u;     // xCalcHADs8x8 rounding
#pragma unroll
      for (int m = 1; m < SEG; m <<= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
      if (ok && has && (lane & (SEG - 1)) == 0) {
        if (LOG2N >= 4) atomicAdd(acc + (r.ctu * C::PUS + r.pu) * kNumModes + mode, v);
        else acc16[(r.ctu * C::PUS + r.pu) * kNumModes + mode] = (uint16_t)(v >> shift);
      }
    }
  };

  // ---- static operands of the pass: the row's source tile (A of the -H product), the constant window slots -----------
  {
    uint4* d = reinterpret_cast<uint4*>(sAorg + rowChunk);
#pragma unroll
    for (int i = 0; i < 8; i++) d[i * 128] = make_uint4(p[4 * i], p[4 * i + 1], p[4 * i + 2], p[4 * i + 3]);
    if (LOG2N != 2) reinterpret_cast<uint4*>(sA1 + rowChunk)[3 * 128] = make_uint4(0u, 0u, 0u, kConstWord);
  }
  fetch_weights(8, 32);
  // round 0 prediction: planar (true orientation rows) / DC (transposed rows) on the ALU
  const unsigned char* unfMain = store + arr_k0_off<LOG2N>(grp, slot, r.o, 0);
  const unsigned char* unfSide = store + arr_k0_off<LOG2N>(grp, slot, r.o ^ 1, 0);
  if (ok) {
    if (LOG2N == 2) { if (r.o == 0) planar_region16(rec, p); else dc_region16(rec, p); }
    else if (r.o == 0) {
      constexpr int f = C::HAS_FILT ? 1 : 0;        // planar reads the smoothed border for N = 8, 16, 32 (TComPattern.cpp:523-548)
      planar_tile16(LOG2N, store + arr_k0_off<LOG2N>(grp, slot, 0, f), store + arr_k0_off<LOG2N>(grp, slot, 1, f), r.u0, r.v0, p);
    } else {
      dc_tile16((reinterpret_cast<const int*>(smem + C::DC_OFF)[r.ctu * 64 + r.pu] + N) >> (LOG2N + 1), C::EDGE, unfMain, unfSide, r.u0, r.v0, p);
    }
  }
  fence_async_smem();                               // the source operand is read by the tensor core (async proxy)

  // ---- round 0 -------------------------------------------------------------------------------------------------
  store_a2(p);
  issue_mma2();
  stage_window(8, 32);
  wait_mma2();
  issue_mma1();
  cost_out(r.o ? 1 : 0, true);

  // ---- angular rounds -----------------------------------------------------------------------------------------
  int angleNext = 26;
#pragma unroll 1
  for (int am = 8; am >= -8; --am) {
    const int angleNext2 = am > -7 ? angle_of_am(am - 2) : 0;
    wait_mma1();
    if (am > -8) fetch_weights(am - 1, angleNext);
    // epilogue 1: the low 16 bits of every accumulator hold 32768 + 32 * pred + remainder
    {
      uint32_t v[32];
      tmem_ld16_pack(tD1 + laneOff, v);
      tmem_ld16_pack(tD1 + laneOff + 32, v + 16);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 32; i++) p[i] = pack_pred16(v[i]);
    }
    if (C::EDGE && am == 0 && ok) {
      if (LOG2N == 2) patch_edge0_region16(rec, maxVal, p);
      else if (r.u0 == 0) patch_edge0_tile16(unfMain, unfSide, r.v0, maxVal, p);
    }
    store_a2(p);
    // projected samples of the next (negative) angle; ordering argument as in tc2_pass: a window that may read another row's
    // projected samples is gathered after wait_mma2 (MMA 2 is only issued once every row has announced arrA, which a row
    // does after writing its projected samples)
    const bool lateWindow = LOG2N != 2 && am > -8 && angleNext < 0;
    if (lateWindow) build_ext_group16<LOG2N>(rowTid, grp, inv_angle_of_am(am - 1), mode_uses_filtered<LOG2N>(25 + am) ? 1 : 0, store);
    arrive_mma2();
    fire_mma2();
    if (am > -8 && !lateWindow) stage_window(am - 1, angleNext);
    wait_mma2();
    if (lateWindow) stage_window(am - 1, angleNext);
    if (am > -8) issue_mma1();
    cost_out(r.o ? 10 - am : 26 + am, !(r.o && am == -8));
    angleNext = angleNext2;
  }
}

template <int LOG2N>
__device__ __noinline__ void tc3_body(const Tc3Args& a, const int unit) {
  typedef Cfg<LOG2N> C;
  unsigned char* smem = smem3;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int shift = a.bitDepth - 8;
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  if (a.fs.needed) {
    // fork-aware mode: a CTA none of whose PUs has to be evaluated writes the table codes and leaves
    if (!__syncthreads_or(fork_states<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, tid, kThreads))) {
      copy_out<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, false, CostRead<LOG2N>{acc, shift}, tid, kThreads);
      return;
    }
    __syncthreads();
  }
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::BAR_OFF);
  uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(smem + C::BAR_OFF + 96);
  if (tid == 0) {
    for (int i = 0; i < 5 * kGroups; i++) mbar_init(bars + i, (i >= 2 * kGroups && i < 4 * kGroups) ? 128 : 1);   // MMA done x2, operands ready x2, weights landed
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) tmem_alloc(tmemSlot, 256);
  // Every global load of the set-up is issued here, before anything waits: the Hadamard operand, the reconstruction
  // neighbourhoods of the CTA's CTUs and the rows' source tiles of pass 0 share ONE memory round trip.
  constexpr int HAD_V = C::HAD_BYTES / 16;         // 512 (two per thread) or 32
  uint4 hadV[2] = {make_uint4(0u, 0u, 0u, 0u), make_uint4(0u, 0u, 0u, 0u)};
  {
    const uint4* h = reinterpret_cast<const uint4*>(a.had + (LOG2N == 2 ? 8192 : 0));
    if (tid < HAD_V) hadV[0] = h[tid];
    if (tid + kThreads < HAD_V) hadV[1] = h[tid + kThreads];
  }
  int ctuX[C::CTUS], ctuY[C::CTUS];
  TileLoad tl[C::CTUS];
  Vec16 pre[8];
  setup_loads<Cfg, LOG2N>(a.fs, unit, a.totalCtus, tid, ctuX, ctuY, tl, pre);
  // every byte a window, a record or an accumulator update may touch starts as zero (finite operands; sums for N >= 16)
  {
    const uint4 z = make_uint4(0u, 0u, 0u, 0u);
    uint4* s = reinterpret_cast<uint4*>(smem + C::STORE_OFF);
    for (int i = tid; i < (C::TOTAL - C::STORE_OFF) / 16; i += kThreads) s[i] = z;          // store + cost accumulators
    if (LOG2N == 2) {
      uint4* r4 = reinterpret_cast<uint4*>(smem + C::A1_OFF);
      for (int i = tid; i < kGroups * C::A1_BYTES / 16; i += kThreads) r4[i] = z;           // records of PUs outside the picture
    }
    reinterpret_cast<int*>(smem + C::DC_OFF)[tid] = 0;          // CTUS * 64 <= 256 sums
  }
  if (tid < HAD_V) reinterpret_cast<uint4*>(smem + C::HAD_OFF)[tid] = hadV[0];
  if (tid + kThreads < HAD_V) reinterpret_cast<uint4*>(smem + C::HAD_OFF)[tid + kThreads] = hadV[1];
  __syncthreads();
  tc3_prologue<LOG2N>(a, unit, tl, ctuX, ctuY);
  __syncthreads();
  // (N >= 8: the tiles aliased the window and source operands; every row rewrites all of its operand chunks before the first MMA)
  tc_fence_before();
  fence_async_smem();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmemBase = *tmemSlot;
  uint32_t ph1 = 0, ph2 = 0, phA = 0, phB = 0, phT = 0;
#pragma unroll 1
  for (int pass = 0; pass < C::PASSES; pass++) tc3_pass<LOG2N>(a, unit, pass, tmemBase, ph1, ph2, phA, phB, phT, pre);

  // ---- costs leave the SM ------------------------------------------------------------------------------------
  tc_fence_before();
  // the common case - every PU of the CTA evaluated - copies the accumulators without a per-element state look-up
  const bool allEval = __syncthreads_and(all_evaluated<Cfg, LOG2N>(smem + C::VALID_OFF, tid, kThreads)) && unit * C::CTUS + C::CTUS <= a.totalCtus;
  copy_out<Cfg, LOG2N>(a.fs, unit, a.totalCtus, smem + C::VALID_OFF, allEval, CostRead<LOG2N>{acc, shift}, tid, kThreads);
  if (warp == 0) tmem_dealloc(tmemBase, 256);
}

// blocks of one launch: depth-major (rmd_tc_frame.cuh frame_block)
__global__ void __launch_bounds__(kThreads, 2)
rmd_frame_tc3_kernel(const __grid_constant__ Tc3Args a) {
  const FrameBlock fb = frame_block(a.totalCtus, blockIdx.x);
  switch (fb.log2n) {
    case 6: tc3_body<6>(a, fb.unit); break;
    case 5: tc3_body<5>(a, fb.unit); break;
    case 4: tc3_body<4>(a, fb.unit); break;
    case 3: tc3_body<3>(a, fb.unit); break;
    default: tc3_body<2>(a, fb.unit);
  }
}

}  // namespace

int rmd_tc3_smem_bytes() { return kSmemBytes; }

cudaError_t configure_rmd_tc3_kernels() {
  return cudaFuncSetAttribute(rmd_frame_tc3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes);
}

cudaError_t launch_rmd_frames_tc3(const FrameSource& fs, int nPics, int bitDepth, int strong, const uint8_t* tabWin16, const uint8_t* tabN416,
                                  const uint8_t* hadamard16, cudaStream_t st, int* launches) {
  const int total = nPics * fs.ctusPerPic;
  if (total <= 0) return cudaSuccess;
  Tc3Args a;
  a.fs = fs; a.strong = strong; a.totalCtus = total; a.bitDepth = bitDepth; a.tabWin = tabWin16; a.tabN4 = tabN416; a.had = hadamard16;
  rmd_frame_tc3_kernel<<<frame_blocks(total), kThreads, kSmemBytes, st>>>(a);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace cucd
