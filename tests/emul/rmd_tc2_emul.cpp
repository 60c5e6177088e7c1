// rmd_tc2_emul.cpp - CPU replay of the tensor-core RMD frame kernel (TEST HARNESS, not a product path).
//
// Compiles csrc/rmd_tc2.cuh (the kernel's __host__ __device__ logic: weight tables, row map, window
// gather, byte packing, planar/DC, border conversion) and csrc/rmd_tc_frame.cuh (block decode, PU states, set-up
// loads, tile staging, copy-out) with g++ and replays one CTA of rmd_tc2_kernels.cu phase by phase for all 256
// worker thread ids.  The two tcgen05 products are replaced by exact integer matmuls
// that read their operands through the same UMMA shared-memory layout / TMEM row layout the kernel uses,
// and tcgen05.ld.pack::16b by its measured behaviour (profiles/ubench).  Built only by tests/.
//
// Frame mode builds the CTA's reference arrays in one of two ways: with the in-CTA prologue the kernel ran before its border pre-pass
// existed (tile_store + build_unfiltered + build_filtered, emul_rmd_frame_tc2), or as the GPU does now, from the images of the replayed
// pre-pass (tests/emul/tc2_prep_replay.h) placed by the CTA's bulk copies (emul_rmd_frames_tc2_prep).
#include <cstdint>
#include <cstring>
#include <type_traits>
#include <vector>
#include "rmd_tc2.cuh"
#include "rmd_tc_frame.cuh"
#include "tc2_prep_replay.h"

using namespace cucd;
using namespace cucd::tc2;
using namespace cucd::tcf;

namespace {

struct Tables {
  std::vector<uint8_t> win, n4;
  std::vector<int8_t> had;   // +H8(x)H8 at 0, block-diagonal +H4(x)H4 at 8192 (layout of hadamard_operands_kernel)
  Tables() : win(kWinTableBytes), n4(kN4TableBytes), had(16384, 0) {
    fill_win_tables(win.data()); fill_n4_tables(n4.data());
    for (int j = 0; j < 64; j++)
      for (int k = 0; k < 64; k++) {
        const int y = k >> 3, x = k & 7, off = umma_off64(j, k);
        const int s8 = (__builtin_popcount((j >> 3) & y) + __builtin_popcount((j & 7) & x)) & 1;
        had[off] = (int8_t)(s8 ? -1 : 1); had[4096 + off] = (int8_t)(s8 ? 1 : -1);
        const int q = j >> 4, u = (j >> 2) & 3, v = j & 3, qk = (y >> 2) * 2 + (x >> 2);
        const int s4 = (__builtin_popcount(u & (y & 3)) + __builtin_popcount(v & (x & 3))) & 1;
        const int e = q == qk ? (s4 ? -1 : 1) : 0;
        had[8192 + off] = (int8_t)e; had[12288 + off] = (int8_t)(-e);
      }
  }
};
const Tables& tables() { static Tables t; return t; }

// D[row][j] = sum_k A[row][k] * B[j][k];  A: bytes of `words` (K/4 words per row), B: UMMA layout, u8 or s8
void mma(const uint32_t* aWords, int aStride, int K, const void* b, bool bSigned, uint32_t* d /*[128][64]*/) {
  for (int row = 0; row < 128; row++)
    for (int j = 0; j < 64; j++) {
      int32_t s = 0;
      for (int k = 0; k < K; k++) {
        const int av = (aWords[row * aStride + (k >> 2)] >> (8 * (k & 3))) & 0xff;
        const int bv = bSigned ? (int)reinterpret_cast<const int8_t*>(b)[umma_off64(j, k)] : (int)reinterpret_cast<const uint8_t*>(b)[umma_off64(j, k)];
        s += av * bv;
      }
      d[row * 64 + j] = (uint32_t)s;
    }
}

// bs == nullptr: frame (replay) mode; otherwise batch (S2) mode over the PUs of one size described by *bs.  Frame mode with img: the store
// and the DC sums come from the pre-pass images img (kPrepCtuBytes per CTU of the launch), as rmd_frame_tc2_kernel takes them
template <int LOG2N>
void emul_cta(const FrameSource& fs, int strong, int totalCtus, int unit, const BatchSource* bs = nullptr, const uint8_t* img = nullptr) {
  typedef Geo<LOG2N> G;
  typedef Cfg<LOG2N> C;
  constexpr int N = G::N, log2n = LOG2N;
  const Tables& tb = tables();
  std::vector<unsigned char> smemStore(C::TOTAL + 256, 0xA5);
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smemStore.data()) + 127) & ~uintptr_t(127));
  uint32_t* acc = reinterpret_cast<uint32_t*>(smem + C::ACC_OFF);
  uint8_t* valid = smem + C::VALID_OFF;
  if (!bs && fs.needed && !fork_states<Cfg, LOG2N>(fs, unit, totalCtus, valid, 0, 1)) {   // fork-aware early exit (tc2_body)
    copy_out<Cfg, LOG2N>(fs, unit, totalCtus, valid, false, CostRead<LOG2N>{acc}, 0, 1);
    return;
  }
  if (LOG2N >= 4) for (int i = 0; i < C::CTUS * C::PUS * kNumModes; i++) acc[i] = 0;
  if (!img) for (int i = 0; i < C::CTUS * 64; i++) reinterpret_cast<int*>(smem + C::DC_OFF)[i] = 0;   // image mode: copied in
  std::vector<Vec16> pre(kThreads * 8);            // frame mode: the rows' source tiles of pass 0 (setup_loads)
  // ---- prologue (tc2_prologue) ----
  if (bs) {
    constexpr int TPP = 256 / C::PUS;
    for (int c = 0; c < C::CTUS; c++) {
      const int first = (unit * C::CTUS + c) * C::PUS;
      for (int p = 0; p < C::PUS; p++) smem[C::VALID_OFF + c * 256 + p] = first + p < bs->count ? 1 : 0;
    }
    for (int c = 0; c < C::CTUS; c++)
      for (int tid = 0; tid < kThreads; tid++) {
        const int idx = (unit * C::CTUS + c) * C::PUS + tid / TPP;
        build_unfiltered_batch<LOG2N>(tid, c, idx < bs->count ? bs->border + (size_t)bs->pus[idx].borderOff : nullptr, smem);
      }
    for (int c = 0; c < C::CTUS; c++)
      if ((unit * C::CTUS + c) * C::PUS < bs->count) for (int tid = 0; tid < kThreads; tid++) build_filtered<LOG2N>(tid, c, strong, smem);
  } else {
  int ctuXs[C::CTUS], ctuYs[C::CTUS];
  TileLoad tl[C::CTUS];                            // (phase 1 is replayed below by stage_tile)
  for (int tid = 0; tid < kThreads; tid++) setup_loads<Cfg, LOG2N>(fs, unit, totalCtus, tid, ctuXs, ctuYs, img ? nullptr : tl, &pre[tid * 8]);
  for (int c = 0; c < C::CTUS; c++) {
    if (ctuXs[c] < 0) { for (int p = 0; p < G::PUS; p++) valid[c * 256 + p] = kPuOutside; continue; }
    const uint8_t* need = ctu_needed<LOG2N>(fs, unit * C::CTUS + c);
    for (int p = 0; p < G::PUS; p++) valid[c * 256 + p] = pu_state<LOG2N>(fs, need, ctuXs[c], ctuYs[c], p);
  }
  if (img) {
    tc2replay::place_images<LOG2N>(img, unit, totalCtus, smem);
  } else {
  for (int c = 0; c < C::CTUS; c++)          // phase 1: every thread id's tile_load + tile_store
    if (ctuXs[c] >= 0) stage_tile<LOG2N>(0, 1, fs.rec + (size_t)ctu_pos(fs, unit * C::CTUS + c).pic * fs.recPicStride, fs.recStride, fs.W, fs.H, ctuXs[c], ctuYs[c], smem + C::TILE_OFF + c * C::TILE_BYTES);
  for (int c = 0; c < C::CTUS; c++)
    if (ctuXs[c] >= 0) for (int tid = 0; tid < kThreads; tid++) build_unfiltered<LOG2N>(tid, c, fs.W, fs.H, ctuXs[c], ctuYs[c], smem + C::TILE_OFF + c * C::TILE_BYTES, smem);
  for (int c = 0; c < C::CTUS; c++)
    if (ctuXs[c] >= 0) for (int tid = 0; tid < kThreads; tid++) build_filtered<LOG2N>(tid, c, strong, smem);
  }
  }
  std::memset(smem + C::TILE_OFF, 0x5A, C::CTUS * C::TILE_BYTES);   // the tiles alias the operand buffers: gone after the prologue
  unsigned char* store = smem + C::STORE_OFF;
  const int8_t* had = tb.had.data() + (log2n == 2 ? 8192 : 0);
  for (int pass = 0; pass < C::PASSES; pass++) {
    // ---- tc2_pass ----
    std::vector<Row> rows(kThreads); std::vector<char> ok(kThreads);
    std::vector<uint32_t> P(kThreads * 16), A1(kThreads * 16, 0xA5A5A5A5u), D(kThreads * 64);
    for (int tid = 0; tid < kThreads; tid++) {
      const Row r = rows[tid] = row_map<LOG2N>(tid, pass);
      const int cg = unit * C::CTUS + r.ctu;
      ok[tid] = valid[r.ctu * 256 + (log2n == 2 ? 4 * r.pu : r.pu)] == kPuEvaluate;
      uint32_t* p = &P[tid * 16];
      if (ok[tid]) {
        uint32_t raw[16];
        auto pack4 = [](const int16_t* q) { uint32_t w = 0; for (int i = 0; i < 4; i++) w |= (uint32_t)(q[i] & 0xff) << (8 * i); return w; };
        if (!bs) {
          int tx, ty;
          const int16_t* src = frame_src_ptr<LOG2N>(fs, r, cg, tx, ty);
          for (int y = 0; y < 8; y++) {
            const Vec16 v = pass == 0 ? pre[tid * 8 + y] : *reinterpret_cast<const Vec16*>(src + (size_t)y * fs.orgStride);
            raw[2 * y] = bperm(v.x, v.y, 0x6420); raw[2 * y + 1] = bperm(v.z, v.w, 0x6420);
          }
        } else {
          const int first = cg * C::PUS;
          if (log2n == 2) {
            for (int q = 0; q < 4; q++) {
              const int idx = first + 4 * r.pu + q;
              for (int y = 0; y < 4; y++) raw[2 * ((q >> 1) * 4 + y) + (q & 1)] = idx < bs->count ? pack4(bs->org + (size_t)bs->pus[idx].orgOff + 4 * y) : 0u;
            }
          } else {
            const int16_t* src = bs->org + (size_t)bs->pus[first + r.pu].orgOff + (r.o ? r.u0 : r.v0) * N + (r.o ? r.v0 : r.u0);
            for (int y = 0; y < 8; y++) for (int h = 0; h < 2; h++) raw[2 * y + h] = pack4(src + y * N + 4 * h);
          }
        }
        if (r.o) tile_transpose_bytes(raw, p, log2n != 2); else std::memcpy(p, raw, sizeof(raw));
      } else std::memset(p, 0, 64);
    }
    // MMA 2: D = source x -H (the static shared-memory operand) + prediction x +H, accumulated in TMEM
    std::vector<uint32_t> ORG = P, DN(kThreads * 64);
    auto hadamard = [&]() {
      for (int grp = 0; grp < kGroups; grp++) {
        mma(&ORG[grp * 128 * 16], 16, 64, had + 4096, true, &DN[grp * 128 * 64]);
        mma(&P[grp * 128 * 16], 16, 64, had, true, &D[grp * 128 * 64]);
      }
      for (size_t i = 0; i < D.size(); i++) D[i] += DN[i];
    };
    auto cost_out = [&](int am, bool angular) {
      // warps in order; the shuffle reduction over SEG lanes and the shared-memory atomics become a plain sum
      for (int tid = 0; tid < kThreads; tid++) {
        const Row& r = rows[tid];
        const int mode = angular ? (r.o ? 10 - am : 26 + am) : (r.o ? 1 : 0);
        const bool has = !(angular && r.o && am == -8);
        uint32_t q[4];
        for (int c = 0; c < 4; c++) { uint32_t s = 0; for (int k = 0; k < 16; k++) s = sad_acc(D[tid * 64 + c * 16 + k], 0u, s); q[c] = s; }
        const int cg = unit * C::CTUS + r.ctu;
        if (log2n == 2) {
          if (ok[tid] && has) for (int c = 0; c < 4; c++) reinterpret_cast<uint16_t*>(acc)[(r.ctu * C::PUS + 4 * r.pu + c) * kNumModes + mode] = (uint16_t)((q[c] + 1u) >> 1);
        } else if (ok[tid] && has) {
          uint32_t& dst = acc[(r.ctu * C::PUS + r.pu) * kNumModes + mode];
          const uint32_t t = (q[0] + q[1] + q[2] + q[3] + 2u) >> 2;
          if (LOG2N >= 4) dst += t; else dst = t;
        }
      }
    };
    if (log2n == 2)
      for (int tid = 0; tid < kThreads; tid++) std::memcpy(&A1[tid * 16], store + rec_off(rows[tid].ctu, rows[tid].o, 4 * rows[tid].pu), 64);
    // round 0
    for (int tid = 0; tid < kThreads; tid++) {
      if (!ok[tid]) continue;
      const Row& r = rows[tid]; uint32_t* p = &P[tid * 16];
      const unsigned char* rec4 = store + rec_off(r.ctu, r.o, 4 * r.pu);
      const int grp = tid >> 7, slot = pu_slot2<LOG2N>(r.ctu, r.pu);
      constexpr int f = C::HAS_FILT ? 1 : 0;
      if (log2n == 2) { if (r.o == 0) planar_region4(rec4, p); else dc_region4(rec4, p); }
      else if (r.o == 0) planar_tile(log2n, store + arr_k0_off<LOG2N>(grp, slot, 0, f), store + arr_k0_off<LOG2N>(grp, slot, 1, f), r.u0, r.v0, p);
      else dc_tile((reinterpret_cast<const int*>(smem + C::DC_OFF)[r.ctu * 64 + r.pu] + N) >> (LOG2N + 1), C::EDGE, store + arr_k0_off<LOG2N>(grp, slot, 1, 0),
                   store + arr_k0_off<LOG2N>(grp, slot, 0, 0), r.u0, r.v0, p);
    }
    hadamard();
    cost_out(0, false);
    for (int am = 8; am >= -8; --am) {
      const int angle = angle_of_am(am), ai = am + 8;
      const int filt = mode_uses_filtered<LOG2N>(26 + am) ? 1 : 0;
      if (log2n != 2 && angle < 0) for (int tid = 0; tid < kThreads; tid++) build_ext_group<LOG2N>(tid & 127, tid >> 7, inv_angle_of_am(am), filt, store);
      for (int grp = 0; grp < kGroups; grp++) {
        const uint8_t* b1;
        if (log2n == 2) b1 = tb.n4.data() + ai * 4096;
        else {
          b1 = tb.win.data() + (ai * 4 + (group_frac0<LOG2N>(grp, pass, angle) >> 3)) * 2048;
          for (int rt = 0; rt < 128; rt++) {
            const int tid = grp * 128 + rt; const Row& r = rows[tid];
            gather_window(store, arr_k0_off<LOG2N>(grp, pu_slot2<LOG2N>(r.ctu, r.pu), r.o, filt) + win_k0(angle, r.u0, r.v0), &A1[tid * 16]);
          }
        }
        mma(&A1[grp * 128 * 16], 16, log2n == 2 ? 64 : 32, b1, false, &D[grp * 128 * 64]);
      }
      for (int tid = 0; tid < kThreads; tid++) {
        const Row& r = rows[tid]; uint32_t* p = &P[tid * 16];
        for (int h = 0; h < 2; h++) {
          uint32_t v[16];
          for (int j = 0; j < 16; j++) v[j] = (D[tid * 64 + h * 32 + 2 * j] & 0xffffu) | (D[tid * 64 + h * 32 + 2 * j + 1] << 16);   // tcgen05.ld.pack::16b
          pack_pred(v, p + 8 * h, 8);
        }
        if (C::EDGE && am == 0 && ok[tid]) {
          if (log2n == 2) patch_edge0_region4(store + rec_off(r.ctu, r.o, 4 * r.pu), p);
          else if (r.u0 == 0) {
            const int slot = pu_slot2<LOG2N>(r.ctu, r.pu);
            patch_edge0_tile(store + arr_k0_off<LOG2N>(tid >> 7, slot, r.o, 0), store + arr_k0_off<LOG2N>(tid >> 7, slot, r.o ^ 1, 0), r.v0, p);
          }
        }
      }
      hadamard();
      cost_out(am, true);
    }
  }
  if (bs) {
    for (int i = 0; i < C::CTUS * C::PUS * kNumModes; i++) {
      const int pl = i / kNumModes, m = i - pl * kNumModes, idx = unit * C::CTUS * C::PUS + pl;
      if (idx >= bs->count) continue;
      bs->out[(size_t)bs->pus[idx].outIndex * kNumModes + m] = CostRead<LOG2N>{acc}(0, i);
    }
    return;
  }
  copy_out<Cfg, LOG2N>(fs, unit, totalCtus, valid, all_evaluated<Cfg, LOG2N>(valid, 0, 1) && unit * C::CTUS + C::CTUS <= totalCtus, CostRead<LOG2N>{acc}, 0, 1);
}

}  // namespace

extern "C" {

// 8-bit frame (replay) mode over ALL CTUs of one picture, as rmd_frame_tc2_kernel writes it; needed: [ctu][341] fork-aware mask or null
int emul_rmd_frame_tc2(int strong, const int16_t* org, int orgStride, const int16_t* rec, int recStride, int W, int H, uint32_t* out, const uint8_t* needed) {
  FrameSource fs;
  fs.org = org; fs.rec = rec; fs.orgPicStride = 0; fs.recPicStride = 0; fs.orgStride = orgStride; fs.recStride = recStride;
  fs.W = W; fs.H = H; fs.ctusPerRow = (W + 63) / 64; fs.ctusPerPic = fs.ctusPerRow * ((H + 63) / 64); fs.out = out; fs.outPacked = nullptr; fs.needed = needed;
  const int total = fs.ctusPerPic;
  for (int b = 0; b < frame_blocks(total); b++) {
    const FrameBlock fb = frame_block(total, b);
    switch (fb.log2n) {
      case 6: emul_cta<6>(fs, strong, total, fb.unit); break;
      case 5: emul_cta<5>(fs, strong, total, fb.unit); break;
      case 4: emul_cta<4>(fs, strong, total, fb.unit); break;
      case 3: emul_cta<3>(fs, strong, total, fb.unit); break;
      default: emul_cta<2>(fs, strong, total, fb.unit);
    }
  }
  return 0;
}
// The frame path the GPU runs: the border pre-pass over nPics pictures (picture p at org + p * orgPicStride, rec + p * recPicStride)
// into an image buffer that holds `poison` everywhere before it runs (what an earlier launch left in the scratch), then every CTA of the
// launch on the images.  needed: [ctu][341] fork-aware mask of the launch or null; out: [nPics * ctusPerPic][341][35]
int emul_rmd_frames_tc2_prep(int strong, int nPics, const int16_t* org, long long orgPicStride, int orgStride, const int16_t* rec, long long recPicStride,
                             int recStride, int W, int H, uint32_t* out, const uint8_t* needed, int poison) {
  FrameSource fs;
  fs.org = org; fs.rec = rec; fs.orgPicStride = orgPicStride; fs.recPicStride = recPicStride; fs.orgStride = orgStride; fs.recStride = recStride;
  fs.W = W; fs.H = H; fs.ctusPerRow = (W + 63) / 64; fs.ctusPerPic = fs.ctusPerRow * ((H + 63) / 64); fs.out = out; fs.outPacked = nullptr; fs.needed = needed;
  const int total = nPics * fs.ctusPerPic;
  const std::vector<uint8_t> img = tc2replay::emul_prep(fs, strong, total, (uint8_t)poison);
  for (int b = 0; b < frame_blocks(total); b++) {
    const FrameBlock fb = frame_block(total, b);
    switch (fb.log2n) {
      case 6: emul_cta<6>(fs, strong, total, fb.unit, nullptr, img.data()); break;
      case 5: emul_cta<5>(fs, strong, total, fb.unit, nullptr, img.data()); break;
      case 4: emul_cta<4>(fs, strong, total, fb.unit, nullptr, img.data()); break;
      case 3: emul_cta<3>(fs, strong, total, fb.unit, nullptr, img.data()); break;
      default: emul_cta<2>(fs, strong, total, fb.unit, nullptr, img.data());
    }
  }
  return 0;
}
// tc2::pu_avail of the PU of size 1 << log2n at (x0, y0): out = {lenL, lenT, availC}
int emul_pu_avail(int log2n, int x0, int y0, int W, int H, int* out) {
  PuAvail a;
  switch (log2n) {
    case 2: a = pu_avail<2>(x0, y0, W, H); break;
    case 3: a = pu_avail<3>(x0, y0, W, H); break;
    case 4: a = pu_avail<4>(x0, y0, W, H); break;
    case 5: a = pu_avail<5>(x0, y0, W, H); break;
    case 6: a = pu_avail<6>(x0, y0, W, H); break;
    default: return -1;
  }
  out[0] = a.lenL; out[1] = a.lenT; out[2] = a.availC;
  return 0;
}
// batch (S2) mode: `count` PUs of ONE size, tightly packed org blocks and borders, out[count][35]
int emul_rmd_batch_tc2(int strong, int log2n, int count, const int16_t* org, const int16_t* border, uint32_t* out) {
  const int n = 1 << log2n, pus = 4096 / (n * n);
  std::vector<BatchPu> list(count);
  for (int i = 0; i < count; i++) { list[i].orgOff = i * n * n; list[i].borderOff = i * (4 * n + 1); list[i].outIndex = i; list[i].pad = 0; }
  BatchSource bs; bs.org = org; bs.border = border; bs.pus = list.data(); bs.out = out; bs.count = count;
  FrameSource fs = {};
  const int units = (count + pus - 1) / pus;
  auto run = [&](auto tag) {
    constexpr int L = decltype(tag)::value;
    for (int u = 0; u * Cfg<L>::CTUS < units; u++) emul_cta<L>(fs, strong, units, u, &bs);
  };
  switch (log2n) {
    case 2: run(std::integral_constant<int, 2>()); break;
    case 3: run(std::integral_constant<int, 3>()); break;
    case 4: run(std::integral_constant<int, 4>()); break;
    case 5: run(std::integral_constant<int, 5>()); break;
    case 6: run(std::integral_constant<int, 6>()); break;
    default: return -1;
  }
  return 0;
}
// the weight tables, for inspection
int emul_tc2_tables(uint8_t* win, uint8_t* n4) { fill_win_tables(win); fill_n4_tables(n4); return 0; }

}  // extern "C"
