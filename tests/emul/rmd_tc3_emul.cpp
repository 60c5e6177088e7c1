// rmd_tc3_emul.cpp - CPU replay of the half-precision tensor-core RMD frame kernel (TEST HARNESS, not a product path).
//
// Compiles csrc/rmd_tc3.cuh (the kernel's __host__ __device__ logic: fp16 weight tables, shared-memory layout, window
// gather, record layout of the N = 4 path, planar / DC, border construction) and csrc/rmd_tc_frame.cuh (block decode, PU
// states, set-up loads, tile staging, copy-out) with g++ and replays one CTA of
// rmd_tc3_kernels.cu phase by phase for all 256 thread ids.  The tcgen05 kind::f16 products are replaced by products of the
// decoded half-precision operands read through the same UMMA shared-memory layout, accumulated in double and rounded to
// fp32 once (every intermediate is an integer below 2^24, so any accumulation order gives this value), and
// tcgen05.ld.pack::16b by the low 16 bits of the fp32 bit pattern (profiles/ubench).  Built only by tests/.
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#include "rmd_tc3.cuh"
#include "rmd_tc_frame.cuh"

using namespace cucd;
using namespace cucd::tc3;
using namespace cucd::tcf;

namespace {

double h2d(uint16_t h) {
  const int s = h >> 15, e = (h >> 10) & 31, m = h & 1023;
  double v;
  if (e == 31) v = NAN;                       // Inf / NaN: poison
  else if (e == 0) v = std::ldexp((double)m, -24);
  else v = std::ldexp((double)(1024 + m), e - 25);
  return s ? -v : v;
}
uint32_t f32_bits(double d) { const float f = (float)d; uint32_t u; std::memcpy(&u, &f, 4); return u; }
float bits_f32(uint32_t u) { float f; std::memcpy(&f, &u, 4); return f; }

struct Tables16 {
  std::vector<uint8_t> win, n4, had;
  Tables16() : win(kWinTableBytes16), n4(kN4TableBytes16), had(kHadBytes16) {
    fill_win_tables16(win.data()); fill_n4_tables16(n4.data()); fill_had_tables16(had.data());
  }
};
const Tables16& tables16() { static Tables16 t; return t; }
uint16_t rd16(const unsigned char* p) { return (uint16_t)(p[0] | (p[1] << 8)); }

template <int LOG2N>
void emul_cta3(const FrameSource& fs, int strong, int bitDepth, int totalCtus, int unit) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, log2n = LOG2N, NB = LOG2N == 2 ? 16 : 64;
  const Tables16& tb = tables16();
  const int maxVal = (1 << bitDepth) - 1, shift = bitDepth - 8;
  std::vector<unsigned char> smemStore(C::TOTAL + 256, 0xFF);          // 0xFFFF is a NaN: stale bytes poison the result
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smemStore.data()) + 127) & ~uintptr_t(127));
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  uint16_t* acc16 = reinterpret_cast<uint16_t*>(acc);
  uint8_t* valid = smem + C::VALID_OFF;
  if (fs.needed && !fork_states<Cfg, LOG2N>(fs, unit, totalCtus, valid, 0, 1)) {   // fork-aware early exit (tc3_body)
    copy_out<Cfg, LOG2N>(fs, unit, totalCtus, valid, false, CostRead<LOG2N>{acc, shift}, 0, 1);
    return;
  }
  // ---- tc3_body set-up ----
  std::memcpy(smem + C::HAD_OFF, tb.had.data() + (log2n == 2 ? 8192 : 0), C::HAD_BYTES);
  std::memset(smem + C::STORE_OFF, 0, C::TOTAL - C::STORE_OFF);
  if (log2n == 2) std::memset(smem + C::A1_OFF, 0, kGroups * C::A1_BYTES);
  for (int i = 0; i < 256; i++) reinterpret_cast<int*>(smem + C::DC_OFF)[i] = 0;
  int ctuXs[C::CTUS], ctuYs[C::CTUS];
  TileLoad tl[C::CTUS];                                                // (phase 1 is replayed below by stage_tile16)
  std::vector<Vec16> pre(kThreads * 8);                                // the rows' source tiles of pass 0
  for (int tid = 0; tid < kThreads; tid++) setup_loads<Cfg, LOG2N>(fs, unit, totalCtus, tid, ctuXs, ctuYs, tl, &pre[tid * 8]);
  // ---- tc3_prologue ----
  for (int c = 0; c < C::CTUS; c++) {
    if (ctuXs[c] < 0) { for (int p = 0; p < C::PUS; p++) valid[c * 256 + p] = kPuOutside; continue; }
    const uint8_t* need = ctu_needed<LOG2N>(fs, unit * C::CTUS + c);
    for (int p = 0; p < C::PUS; p++) valid[c * 256 + p] = pu_state<LOG2N>(fs, need, ctuXs[c], ctuYs[c], p);
    stage_tile16<LOG2N>(0, 1, fs.rec + (size_t)ctu_pos(fs, unit * C::CTUS + c).pic * fs.recPicStride, fs.recStride, fs.W, fs.H, ctuXs[c], ctuYs[c],
                        reinterpret_cast<uint16_t*>(smem + C::TILE_OFF + c * C::TILE_BYTES));   // phase 1: every thread id's tile_load + tile_store
  }
  for (int c = 0; c < C::CTUS; c++)
    if (ctuXs[c] >= 0)
      for (int tid = 0; tid < kThreads; tid++)
        build_unfiltered16<LOG2N>(tid, c, fs.W, fs.H, ctuXs[c], ctuYs[c], bitDepth, reinterpret_cast<const uint16_t*>(smem + C::TILE_OFF + c * C::TILE_BYTES), smem);
  for (int c = 0; c < C::CTUS; c++)
    if (ctuXs[c] >= 0) for (int tid = 0; tid < kThreads; tid++) build_filtered16<LOG2N>(tid, c, strong, bitDepth, smem);
  std::memset(smem + C::TILE_OFF, 0xFF, C::CTUS * C::TILE_BYTES);       // the tiles alias operand buffers: gone after the prologue
  unsigned char* store = smem + C::STORE_OFF;

  auto a_elem = [&](int off, int bytesPerGroup, int grp, int row, int k) {   // element k of a row of a 128-row operand in shared memory
    return h2d(rd16(smem + off + grp * bytesPerGroup + (k >> 3) * 2048 + row_chunk(row) + (k & 7) * 2));
  };
  for (int pass = 0; pass < C::PASSES; pass++) {
    std::vector<Row> rows(kThreads); std::vector<char> ok(kThreads);
    std::vector<uint32_t> P(kThreads * 32);              // A2 in TMEM
    std::vector<uint32_t> D(kThreads * 64);              // accumulator bit patterns
    for (int tid = 0; tid < kThreads; tid++) {
      const int grp = tid >> 7, rowTid = tid & 127;
      const Row r = rows[tid] = row_map<LOG2N>(tid, pass);
      const int cg = unit * C::CTUS + r.ctu;
      ok[tid] = valid[r.ctu * 256 + (log2n == 2 ? 4 * r.pu : r.pu)] == kPuEvaluate;
      uint32_t* p = &P[tid * 32];
      if (ok[tid]) {
        uint32_t raw[32];
        int tx, ty;
        const int16_t* src = frame_src_ptr<LOG2N>(fs, r, cg, tx, ty);
        for (int y = 0; y < 8; y++) {
          const Vec16 v = pass == 0 ? pre[tid * 8 + y] : *reinterpret_cast<const Vec16*>(src + (size_t)y * fs.orgStride);
          raw[4 * y] = v.x; raw[4 * y + 1] = v.y; raw[4 * y + 2] = v.z; raw[4 * y + 3] = v.w;
        }
        if (log2n == 2) region_to_quadrants16(raw, p, r.o != 0);
        else if (r.o) tile_transpose16(raw, p);
        else std::memcpy(p, raw, sizeof(raw));
        for (int i = 0; i < 32; i++) p[i] = (p[i] & kMask2) | kBias2;
      } else std::memset(p, 0, 128);
      unsigned char* sAorg = smem + C::AORG_OFF + grp * C::AORG_BYTES + row_chunk(rowTid);
      for (int i = 0; i < 8; i++) std::memcpy(sAorg + i * 2048, p + 4 * i, 16);
      if (log2n != 2) {
        const uint32_t c3[4] = {0u, 0u, 0u, kConstWord};
        std::memcpy(smem + C::A1_OFF + grp * C::A1_BYTES + row_chunk(rowTid) + 3 * 2048, c3, 16);
      }
    }
    // store_a2: A2 = (1024 + pred) - (1024 + src) per half as HSUB2 computes it - exact, because the difference of two fp16
    // integers in [1024, 2048) (or 0 for rows that are not evaluated) is an integer of magnitude <= 2047; then MMA 2: D2 = A2 x H
    auto hsub = [](uint16_t x, uint16_t y) -> uint16_t {
      const double d = h2d(x) - h2d(y);
      const int v = (int)d;
      if ((double)v != d || v < -2048 || v > 2048) return 0x7e00;                 // not exactly representable: poison (NaN)
      return (uint16_t)((v < 0 ? 0x8000 : 0) | h16_of_int(v < 0 ? -v : v));
    };
    auto hadamard = [&]() {
      for (int tid = 0; tid < kThreads; tid++) {
        const int grp = tid >> 7, row = tid & 127;
        uint32_t A2[32];
        for (int w = 0; w < 32; w++) {
          const unsigned char* sp = smem + C::AORG_OFF + grp * C::AORG_BYTES + (w >> 2) * 2048 + row_chunk(row) + (w & 3) * 4;
          const uint32_t pw = P[tid * 32 + w];
          A2[w] = (uint32_t)hsub((uint16_t)(pw & 0xffffu), rd16(sp)) | ((uint32_t)hsub((uint16_t)(pw >> 16), rd16(sp + 2)) << 16);
        }
        for (int j = 0; j < 64; j++) {
          const int q = log2n == 2 ? j >> 4 : 0, jl = log2n == 2 ? j & 15 : j, K = log2n == 2 ? 16 : 64;
          double s = 0;
          for (int k = 0; k < K; k++) {
            const int kk = q * 16 + k;
            const uint32_t w = A2[kk >> 1];
            s += h2d((uint16_t)((kk & 1) ? w >> 16 : w & 0xffffu)) * h2d(rd16(smem + C::HAD_OFF + umma16_off(NB, jl, k)));
          }
          D[tid * 64 + j] = f32_bits(s);
        }
      }
    };
    auto cost_out = [&](int am, bool angular) {
      for (int tid = 0; tid < kThreads; tid++) {
        const Row& r = rows[tid];
        const int mode = angular ? (r.o ? 10 - am : 26 + am) : (r.o ? 1 : 0);
        const bool has = !(angular && r.o && am == -8);
        float q[4];
        for (int c = 0; c < 4; c++) { float s = 0.f; for (int k = 0; k < 16; k++) s += std::fabs(bits_f32(D[tid * 64 + c * 16 + k])); q[c] = s; }
        if (!(ok[tid] && has)) continue;
        if (log2n == 2) {
          for (int c = 0; c < 4; c++) acc16[(r.ctu * C::PUS + 4 * r.pu + c) * kNumModes + mode] = (uint16_t)((((uint32_t)q[c] + 1u) >> 1) >> shift);
        } else {
          const uint32_t t = ((uint32_t)((q[0] + q[1]) + (q[2] + q[3])) + 2u) >> 2;
          if (LOG2N >= 4) acc[(r.ctu * C::PUS + r.pu) * kNumModes + mode] += t;
          else acc16[(r.ctu * C::PUS + r.pu) * kNumModes + mode] = (uint16_t)(t >> shift);
        }
      }
    };
    // round 0
    for (int tid = 0; tid < kThreads; tid++) {
      if (!ok[tid]) continue;
      const Row& r = rows[tid]; uint32_t* p = &P[tid * 32];
      const int grp = tid >> 7, slot = pu_slot<LOG2N>(r.ctu, r.pu);
      auto rec = [&](int q, int s) { return ld_s16(smem + rec_slot_off(r.ctu, r.o, 4 * r.pu + q, s)); };
      constexpr int f = C::HAS_FILT ? 1 : 0;
      if (log2n == 2) { if (r.o == 0) planar_region16(rec, p); else dc_region16(rec, p); }
      else if (r.o == 0) planar_tile16(log2n, store + arr_k0_off<LOG2N>(grp, slot, 0, f), store + arr_k0_off<LOG2N>(grp, slot, 1, f), r.u0, r.v0, p);
      else dc_tile16((reinterpret_cast<const int*>(smem + C::DC_OFF)[r.ctu * 64 + r.pu] + N) >> (LOG2N + 1), C::EDGE, store + arr_k0_off<LOG2N>(grp, slot, 1, 0),
                     store + arr_k0_off<LOG2N>(grp, slot, 0, 0), r.u0, r.v0, p);
    }
    hadamard();
    cost_out(0, false);
    for (int am = 8; am >= -8; --am) {
      const int angle = angle_of_am(am), ai = am + 8;
      const int filt = mode_uses_filtered<LOG2N>(26 + am) ? 1 : 0;
      if (log2n != 2 && angle < 0) for (int tid = 0; tid < kThreads; tid++) build_ext_group16<LOG2N>(tid & 127, tid >> 7, inv_angle_of_am(am), filt, store);
      for (int grp = 0; grp < kGroups; grp++) {
        const uint8_t* b1 = log2n == 2 ? tb.n4.data() + ai * kN4Table16 : tb.win.data() + (ai * 4 + (group_frac0<LOG2N>(grp, pass, angle) >> 3)) * kWinTable16;
        std::memcpy(smem + C::B1_OFF + grp * C::B1_BYTES, b1, C::B1_BYTES);                  // the bulk copy
        if (log2n != 2)
          for (int rt = 0; rt < 128; rt++) {
            const int tid = grp * 128 + rt; const Row& r = rows[tid];
            uint32_t w[12];
            gather_window16(store, arr_k0_off<LOG2N>(grp, pu_slot<LOG2N>(r.ctu, r.pu), r.o, filt) + 2 * win_k0(angle, r.u0, r.v0), w);
            unsigned char* d = smem + C::A1_OFF + grp * C::A1_BYTES + row_chunk(rt);
            std::memcpy(d, w, 16); std::memcpy(d + 2048, w + 4, 16); std::memcpy(d + 4096, w + 8, 16);
          }
        // MMA 1
        for (int rt = 0; rt < 128; rt++)
          for (int j = 0; j < 64; j++) {
            const int q = log2n == 2 ? j >> 4 : 0, jl = log2n == 2 ? j & 15 : j, K = log2n == 2 ? 16 : 32;
            double s = 0;
            for (int k = 0; k < K; k++)
              s += a_elem(C::A1_OFF, C::A1_BYTES, grp, rt, q * 16 + k) * h2d(rd16(smem + C::B1_OFF + grp * C::B1_BYTES + umma16_off(NB, jl, k)));
            D[(grp * 128 + rt) * 64 + j] = f32_bits(s);
          }
      }
      for (int tid = 0; tid < kThreads; tid++) {
        const Row& r = rows[tid]; uint32_t* p = &P[tid * 32];
        for (int i = 0; i < 32; i++) p[i] = pack_pred16((D[tid * 64 + 2 * i] & 0xffffu) | (D[tid * 64 + 2 * i + 1] << 16));   // tcgen05.ld.pack::16b
        if (C::EDGE && am == 0 && ok[tid]) {
          auto rec = [&](int q, int s) { return ld_s16(smem + rec_slot_off(r.ctu, r.o, 4 * r.pu + q, s)); };
          if (log2n == 2) patch_edge0_region16(rec, maxVal, p);
          else if (r.u0 == 0) {
            const int slot = pu_slot<LOG2N>(r.ctu, r.pu);
            patch_edge0_tile16(store + arr_k0_off<LOG2N>(tid >> 7, slot, r.o, 0), store + arr_k0_off<LOG2N>(tid >> 7, slot, r.o ^ 1, 0), r.v0, maxVal, p);
          }
        }
      }
      hadamard();
      cost_out(am, true);
    }
  }
  copy_out<Cfg, LOG2N>(fs, unit, totalCtus, valid, all_evaluated<Cfg, LOG2N>(valid, 0, 1) && unit * C::CTUS + C::CTUS <= totalCtus,
                       CostRead<LOG2N>{acc, shift}, 0, 1);
}

}  // namespace

extern "C" {

// frame (replay) mode over ALL CTUs of one picture, as rmd_frame_tc3_kernel writes it (bit depth 8..10); needed: [ctu][341]
// fork-aware mask or null
int emul_rmd_frame_tc3(int bitDepth, int strong, const int16_t* org, int orgStride, const int16_t* rec, int recStride, int W, int H, uint32_t* out,
                       const uint8_t* needed) {
  FrameSource fs;
  fs.org = org; fs.rec = rec; fs.orgPicStride = 0; fs.recPicStride = 0; fs.orgStride = orgStride; fs.recStride = recStride;
  fs.W = W; fs.H = H; fs.ctusPerRow = (W + 63) / 64; fs.ctusPerPic = fs.ctusPerRow * ((H + 63) / 64); fs.out = out; fs.outPacked = nullptr; fs.needed = needed;
  const int total = fs.ctusPerPic;
  for (int b = 0; b < frame_blocks(total); b++) {
    const FrameBlock fb = frame_block(total, b);
    switch (fb.log2n) {
      case 6: emul_cta3<6>(fs, strong, bitDepth, total, fb.unit); break;
      case 5: emul_cta3<5>(fs, strong, bitDepth, total, fb.unit); break;
      case 4: emul_cta3<4>(fs, strong, bitDepth, total, fb.unit); break;
      case 3: emul_cta3<3>(fs, strong, bitDepth, total, fb.unit); break;
      default: emul_cta3<2>(fs, strong, bitDepth, total, fb.unit);
    }
  }
  return 0;
}
int emul_tc3_smem_bytes() { return kSmemBytes; }

}  // extern "C"
