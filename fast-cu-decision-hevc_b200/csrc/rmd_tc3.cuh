// rmd_tc3.cuh - per-thread logic of the tensor-core RMD frame kernel for 9/10-bit content (sm_100a, tcgen05 kind::f16).
//
// Same decomposition as rmd_tc2.cuh (a thread = one 8x8 tile in one orientation = one TMEM lane; MMA 1 predicts the
// 33 angular modes, MMA 2 is the Hadamard of the residual), carried by half-precision operands with fp32 accumulation,
// every value an integer the format holds exactly:
//   * a sample s (0..1023) is stored as the fp16 number 1024 + s = bit pattern 0x6400 | s (ulp 1 in [1024, 2048));
//   * MMA 1:  D = sum w_i * (1024 + ref_i)  +  2048 * 4096  +  1 * 16      with integer weights (32-f), f  (sum 32)
//               = 2^23 + 32768 + [(32-f)*a + f*b + 16]                       (TComPrediction.cpp:368-383)
//     an fp32 in [2^23, 2^24) has ulp 1, so the low 16 bits of its bit pattern are 32768 + 32*pred + remainder:
//     tcgen05.ld.pack::16b returns two of them per register and pred = (x >> 5) & 0x3ff;
//   * the residual (1024 + pred) - (1024 + src) = pred - src is one HSUB2 per pixel pair and exact in fp16 (|.| <= 1023 < 2048);
//     MMA 2:  D = (pred - src) x H exactly (|.| <= 64 * 1023 < 2^24): no source operand on the tensor-core side;
//     the epilogue sums |D| with FADD |x| (exact: the sum stays below 2^24) and converts once.
// N = 4: a row is an 8x8 region of four PUs; the four quadrants are four N = 16, K = 16 products against ONE 16 x 16
// weight table / H4 (x) H4, so region pixels are ordered quadrant-major: j = q*16 + lv*4 + lu.
// Reference arithmetic: TComPrediction.cpp:278-409 (angular), :300-322 (projection), TComRdCost.cpp:1343-1604 (SATD).
#pragma once
#include "rmd_tc2.cuh"

namespace cucd {
namespace tc3 {

using tc2::Row;
using tc2::RowSeg;
using tc2::row_map;
using tc2::group_frac0;
using tc2::win_lmin;
using tc2::win_k0;
using tc2::angle_of_am;
using tc2::inv_angle_of_am;
using tc2::bperm;
using tc2::n4_slot;
using tc2::PuAvail;
using tc2::pu_avail;
using tc2::kAngles;

constexpr int kThreads = 256;
constexpr int kGroups = 2;
constexpr uint32_t kBias2 = 0x64006400u;     // two fp16 1024.0: OR-ing a sample pair turns it into (1024 + s) pairs
constexpr uint32_t kMask2 = 0x03ff03ffu;
constexpr uint32_t kConstWord = 0x3c006800u; // window slots 30, 31: 2048.0 (x 4096 = 2^23), 1.0 (x 16)
constexpr int kWinSamples = 24;              // samples gathered per window (slots 0..23; the weights touch 0..16)
constexpr int kWinTable16 = 4096;            // one MMA 1 weight operand, N >= 8: 64 pixels x 32 slots fp16
constexpr int kN4Table16 = 512;              // N = 4: 16 pixels x 16 slots
constexpr int kWinTableBytes16 = kAngles * 4 * kWinTable16;
constexpr int kN4TableBytes16 = kAngles * kN4Table16;
constexpr int kHadBytes16 = 8192 + 512;      // +H8 (x) H8 (64 x 64 fp16), then +H4 (x) H4 (16 x 16)

// fp16 bit pattern of an integer 0..2048 (exact)
CUCD_HD uint16_t h16_of_int(int v) {
  if (v == 0) return 0;
  int e = 0;
  while ((2 << e) <= v) e++;
  return (uint16_t)(((15 + e) << 10) | ((v - (1 << e)) << (10 - e)));
}
// byte offset of element (row j, k) of a K-major, no-swizzle fp16 UMMA operand with `rows` rows (16-byte chunks of 8 elements)
CUCD_HD int umma16_off(int rows, int j, int k) { return (k >> 3) * rows * 16 + (j >> 3) * 128 + (j & 7) * 16 + (k & 7) * 2; }

inline void put16(uint8_t* t, int off, uint16_t v) { t[off] = (uint8_t)(v & 0xff); t[off + 1] = (uint8_t)(v >> 8); }
// B operand of MMA 1 for N >= 8: table[(am + 8) * 4 + fc], geometry of tc2::fill_win_tables
inline void fill_win_tables16(uint8_t* dst /*kWinTableBytes16*/) {
  for (int i = 0; i < kWinTableBytes16; i++) dst[i] = 0;
  for (int am = -8; am <= 8; am++)
    for (int fc = 0; fc < 4; fc++) {
      uint8_t* t = dst + ((am + 8) * 4 + fc) * kWinTable16;
      const int a = angle_of_am(am), frac0 = fc * 8, lmin = win_lmin(a, frac0);
      for (int v = 0; v < 8; v++) {
        const int d = frac0 + (v + 1) * a, li = d >> 5, f = d & 31;
        for (int u = 0; u < 8; u++) {
          const int j = v * 8 + u, s = u + li - lmin;
          put16(t, umma16_off(64, j, s), h16_of_int(32 - f));
          if (f) put16(t, umma16_off(64, j, s + 1), h16_of_int(f));
          put16(t, umma16_off(64, j, 30), 0x6c00);   // 4096.0
          put16(t, umma16_off(64, j, 31), 0x4c00);   // 16.0
        }
      }
    }
}
// N = 4: table[am + 8] = 16 PU pixels x 16 record slots (main[0..8] at 0..8, side[1..5] at 9..13, 2048 at 14, 1 at 15)
inline void fill_n4_tables16(uint8_t* dst /*kN4TableBytes16*/) {
  for (int i = 0; i < kN4TableBytes16; i++) dst[i] = 0;
  for (int am = -8; am <= 8; am++) {
    uint8_t* t = dst + (am + 8) * kN4Table16;
    const int a = angle_of_am(am), inv = inv_angle_of_am(am);
    for (int lv = 0; lv < 4; lv++)
      for (int lu = 0; lu < 4; lu++) {
        const int j = lv * 4 + lu, d = (lv + 1) * a, f = d & 31, k = lu + (d >> 5) + 1;
        put16(t, umma16_off(16, j, n4_slot(k, inv)), h16_of_int(32 - f));
        if (f) put16(t, umma16_off(16, j, n4_slot(k + 1, inv)), h16_of_int(f));
        put16(t, umma16_off(16, j, 14), 0x6c00);
        put16(t, umma16_off(16, j, 15), 0x4c00);
      }
  }
}
// B operands of MMA 2: +-1.0; coefficient j = (u, v), pixel k = (y, x): (-1)^(<u,y> + <v,x>)
inline void fill_had_tables16(uint8_t* dst /*kHadBytes16*/) {
  auto pc = [](int v) { int c = 0; while (v) { c += v & 1; v >>= 1; } return c; };
  for (int j = 0; j < 64; j++)
    for (int k = 0; k < 64; k++)
      put16(dst, umma16_off(64, j, k), ((pc((j >> 3) & (k >> 3)) + pc((j & 7) & (k & 7))) & 1) ? 0xbc00 : 0x3c00);
  for (int j = 0; j < 16; j++)
    for (int k = 0; k < 16; k++)
      put16(dst + 8192, umma16_off(16, j, k), ((pc((j >> 2) & (k >> 2)) + pc((j & 3) & (k & 3))) & 1) ? 0xbc00 : 0x3c00);
}

// ---------------------------------------------------------------------------------------------
// shared memory of the CTA (work split as tc2::Cfg: 2 CTUs per CTA, N >= 32: 4 CTUs in two passes)
// ---------------------------------------------------------------------------------------------
// fp16 reference arrays of the N >= 8 path: element k of an array lives at byte  arr + 2 * (N + k),  k = -N .. 2N + 1.
// A window may read up to 23 elements past its first one, i.e. past the end of its array into the next one (or into
// the zeroed tail of the group's store): those slots meet zero weights, they only have to hold FINITE numbers, which
// is why the whole store is zeroed before it is filled.
template <int LOG2N>
struct Cfg {
  static constexpr int al16(int v) { return (v + 15) & ~15; }
  static constexpr int N = 1 << LOG2N;
  static constexpr int PUS = 4096 / (N * N);
  static constexpr int CTUS = LOG2N >= 5 ? 4 : 2;
  static constexpr int PASSES = LOG2N >= 5 ? 2 : 1;
  static constexpr bool HAS_FILT = LOG2N >= 3 && LOG2N <= 5;
  static constexpr int NARR = HAS_FILT ? 4 : 2;
  static constexpr int AS = 3 * N + 2;                             // elements per array (even)
  static constexpr int PU_WORDS = NARR * AS / 2;
  static constexpr int PU_BYTES = 4 * (PU_WORDS + ((PU_WORDS & 1) ? 0 : 1));   // odd number of words: lanes of different PUs hit different banks
  static constexpr int SLOTS = LOG2N == 3 ? 64 : CTUS * PUS;
  static constexpr int GROUP_BYTES = LOG2N == 2 ? 0 : al16(16 + SLOTS * PU_BYTES + 64);
  static constexpr int STORE_BYTES = kGroups * GROUP_BYTES;      // N = 4 keeps its records in the A1 operand itself
  static constexpr int HAD_BYTES = LOG2N == 2 ? 512 : 8192;
  static constexpr int B1_BYTES = LOG2N == 2 ? kN4Table16 : kWinTable16;       // per group, single buffer
  static constexpr int A1_BYTES = LOG2N == 2 ? 16384 : 8192;                   // per group: 128 rows x 64 B windows / 128 B records
  static constexpr int AORG_BYTES = 16384;                                     // per group: 128 rows x 64 source samples
  static constexpr int ACC_ELEM = LOG2N <= 3 ? 2 : 4;             // N = 4, 8: final costs (<= 32 736) as uint16; N >= 16: uint32 sums
  static constexpr bool EDGE = LOG2N <= 4;
  static constexpr int HAD_OFF = 0;
  static constexpr int B1_OFF = HAD_OFF + HAD_BYTES;
  static constexpr int A1_OFF = B1_OFF + kGroups * B1_BYTES;
  static constexpr int AORG_OFF = A1_OFF + kGroups * A1_BYTES;
  static constexpr int BAR_OFF = AORG_OFF + kGroups * AORG_BYTES;  // 5 mbarriers per group, TMEM slot at +96
  static constexpr int VALID_OFF = BAR_OFF + 128;
  static constexpr int DC_OFF = VALID_OFF + CTUS * 256;
  static constexpr int STORE_OFF = DC_OFF + CTUS * 64 * 4;
  static constexpr int ACC_OFF = STORE_OFF + al16(STORE_BYTES);
  static constexpr int TOTAL = ACC_OFF + al16(CTUS * PUS * kNumModes * ACC_ELEM);
  // 16-bit copy of the reconstruction around each CTU while the reference arrays are built.  N >= 8: aliases the window and
  // source operands (first written after the prologue); N = 4: only the source operand (the records are built into A1).
  static constexpr int TILE_OFF = LOG2N == 2 ? AORG_OFF : A1_OFF;
  static constexpr int TILE_PITCH = 68;                            // elements
  static constexpr int TILE_X0 = 8;                                // tile[y][x] = t[y * TILE_PITCH + TILE_X0 + x], x = -1 .. 63
  static constexpr int TILE_TOP = 64 * TILE_PITCH;                 // row y = -1: top[x] = t[TILE_TOP + TILE_X0 + x], x = -1 .. 127
  static constexpr int TILE_BYTES = al16(2 * (TILE_TOP + 8 + 128));
  static_assert(CTUS * TILE_BYTES <= BAR_OFF - TILE_OFF, "tiles must fit the aliased operand buffers");
  static_assert(TOTAL <= 113 * 1024, "two CTAs per SM");
};
constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int kSmemBytes = cmax(cmax(cmax(Cfg<2>::TOTAL, Cfg<3>::TOTAL), cmax(Cfg<4>::TOTAL, Cfg<5>::TOTAL)), Cfg<6>::TOTAL);

template <int LOG2N> CUCD_HD int pu_slot(int ctu, int pu) { return LOG2N == 3 ? pu : ctu * Cfg<LOG2N>::PUS + pu; }
// byte offset (from the start of the store) of element k = 0 of array (slot, o, filt) in row group `grp`'s copy
template <int LOG2N> CUCD_HD int arr_k0_off(int grp, int slot, int o, int filt) {
  typedef Cfg<LOG2N> C;
  return grp * C::GROUP_BYTES + 16 + slot * C::PU_BYTES + ((filt * 2 + o) * C::AS + C::N) * 2;
}
// the row's 16-byte slot inside one 128-row chunk of a UMMA operand
CUCD_HD int row_chunk(int rowTid) { return (rowTid >> 3) * 128 + (rowTid & 7) * 16; }
// N = 4: byte offset inside shared memory of slot s of the record of PU `pu4` (0..255) of CTU `ctu` in orientation o.
// The records ARE the A operand of MMA 1: row = o * 64 + region, record q = pu4 & 3 = chunks 2q, 2q + 1 of the row.
CUCD_HD int rec_slot_off(int ctu, int o, int pu4, int s) {
  const int row = o * 64 + (pu4 >> 2), q = pu4 & 3;
  return Cfg<2>::A1_OFF + ctu * Cfg<2>::A1_BYTES + (2 * q + (s >> 3)) * 2048 + row_chunk(row) + (s & 7) * 2;
}
// the cost of element i (= pu * 35 + mode) of the CTA's CTU c in the accumulators at ACC_OFF: final uint16 costs for N <= 8,
// uint32 sums >> (bitDepth - 8) otherwise
template <int LOG2N> struct CostRead {
  const uint32_t* acc; int shift;
  CUCD_HD uint32_t operator()(int c, int i) const {
    const int e = c * Cfg<LOG2N>::PUS * kNumModes + i;
    return LOG2N <= 3 ? (uint32_t)reinterpret_cast<const uint16_t*>(acc)[e] : acc[e] >> shift;
  }
};
CUCD_HD int ld_s16(const unsigned char* p) { return (int)(*reinterpret_cast<const uint16_t*>(p) & 0x3ffu); }   // sample of a stored 1024 + s

// ---------------------------------------------------------------------------------------------
// 16-bit tiles: w[32], word 4*y + h = pixels (y, 2h), (y, 2h + 1) in the halves
// ---------------------------------------------------------------------------------------------
CUCD_HD uint32_t pack_halves(uint32_t a, uint32_t b, int hi) { return hi ? pack_hi(a, b) : pack_lo(a, b); }
// transpose of the whole 8x8
CUCD_HD void tile_transpose16(const uint32_t* w, uint32_t* d) {
#pragma unroll
  for (int v = 0; v < 8; v++)
#pragma unroll
    for (int h = 0; h < 4; h++) d[4 * v + h] = pack_halves(w[(2 * h) * 4 + (v >> 1)], w[(2 * h + 1) * 4 + (v >> 1)], v & 1);
}
// N = 4: raster 8x8 region -> quadrant-major order (word q*8 + lv*2 + h), each 4x4 PU transposed when `transpose`
CUCD_HD void region_to_quadrants16(const uint32_t* w, uint32_t* d, bool transpose) {
#pragma unroll
  for (int q = 0; q < 4; q++)
#pragma unroll
    for (int lv = 0; lv < 4; lv++)
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const int qy = q >> 1, qx = q & 1;
        d[q * 8 + lv * 2 + h] = transpose ? pack_halves(w[(4 * qy + 2 * h) * 4 + 2 * qx + (lv >> 1)], w[(4 * qy + 2 * h + 1) * 4 + 2 * qx + (lv >> 1)], lv & 1)
                                          : w[(4 * qy + lv) * 4 + 2 * qx + h];
      }
}

// MMA 1 operand of a row (N >= 8): 24 fp16 samples starting at byte address `byteOff` (even) of the store -> 12 words
CUCD_HD void gather_window16(const unsigned char* store, int byteOff, uint32_t* w12) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(store + (byteOff & ~3));
  const uint32_t sel = (byteOff & 2) ? 0x5432u : 0x3210u;
  uint32_t x[13];
#pragma unroll
  for (int j = 0; j < 13; j++) x[j] = s[j];
#pragma unroll
  for (int j = 0; j < 12; j++) w12[j] = bperm(x[j], x[j + 1], sel);
}
// epilogue 1: x = two accumulators' low 16 bits (32768 + 32 * pred + remainder each) -> two (1024 + pred) fp16
CUCD_HD uint32_t pack_pred16(uint32_t x) { return ((x >> 5) & kMask2) | kBias2; }
CUCD_HD int clip_bd(int v, int maxVal) { return v < 0 ? 0 : (v > maxVal ? maxVal : v); }
CUCD_HD uint32_t set_lo16(uint32_t w, int v) { return (w & 0xffff0000u) | (uint32_t)v | 0x6400u; }

// pure vertical / horizontal modes, N <= 16: first column gets the edge filter (TComPrediction.cpp:346-363)
// main/side: byte pointers to element 0 (corner) of the fp16 arrays
CUCD_HD void patch_edge0_tile16(const unsigned char* main0, const unsigned char* side0, int v0, int maxVal, uint32_t* p) {
  const int m1 = ld_s16(main0 + 2), s0 = ld_s16(side0);
#pragma unroll
  for (int v = 0; v < 8; v++) p[4 * v] = set_lo16(p[4 * v], clip_bd(m1 + ((ld_s16(side0 + 2 * (v0 + v + 1)) - s0) >> 1), maxVal));
}
// N = 4 region: `rec(q, s)` = sample in slot s of the record of the region's PU q in the row's orientation
template <class Rec>
CUCD_HD void patch_edge0_region16(Rec rec, int maxVal, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const int m1 = rec(q, 1), s0 = rec(q, 0);
#pragma unroll
    for (int lv = 0; lv < 4; lv++) p[q * 8 + lv * 2] = set_lo16(p[q * 8 + lv * 2], clip_bd(m1 + ((rec(q, 9 + lv) - s0) >> 1), maxVal));
  }
}

// ---------------------------------------------------------------------------------------------
// planar and DC on the integer ALU (2 of the 35 modes); 10-bit sums do not fit 16-bit halves: one pixel per integer
// ---------------------------------------------------------------------------------------------
// TComPrediction.cpp:755-805 for the 8x8 tile at (u0, v0) of an N x N PU.  T, L: byte pointers to element 0.
CUCD_HD void planar_tile16(int log2n, const unsigned char* T, const unsigned char* L, int u0, int v0, uint32_t* p) {
  const int N = 1 << log2n;
  const int tr = ld_s16(T + 2 * (N + 1)), bl = ld_s16(L + 2 * (N + 1));
  int V[8], VS[8];
#pragma unroll
  for (int u = 0; u < 8; u++) {
    const int t = ld_s16(T + 2 * (u0 + u + 1));
    V[u] = (N - 1 - v0) * t + (v0 + 1) * bl; VS[u] = bl - t;
  }
#pragma unroll
  for (int v = 0; v < 8; v++) {
    const int l = ld_s16(L + 2 * (v0 + v + 1)), hs = tr - l;
    int h = (N - 1 - u0) * l + (u0 + 1) * tr + N;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const uint32_t a = (uint32_t)((h + V[2 * j]) >> (log2n + 1)), b = (uint32_t)((h + hs + V[2 * j + 1]) >> (log2n + 1));
      p[4 * v + j] = a | (b << 16) | kBias2;
      h += 2 * hs;
    }
#pragma unroll
    for (int u = 0; u < 8; u++) V[u] += VS[u];
  }
}
// TComPrediction.cpp:183-222, 818-841
CUCD_HD void dc_tile16(int dc, bool edge, const unsigned char* main0, const unsigned char* side0, int u0, int v0, uint32_t* p) {
  const uint32_t dc2 = (uint32_t)dc * 0x00010001u | kBias2;
#pragma unroll
  for (int i = 0; i < 32; i++) p[i] = dc2;
  if (!edge) return;
  if (v0 == 0) {
#pragma unroll
    for (int h = 0; h < 4; h++) {
      uint32_t w = 0;
#pragma unroll
      for (int e = 0; e < 2; e++) {
        const int u = 2 * h + e;
        int val = (ld_s16(main0 + 2 * (u0 + u + 1)) + 3 * dc + 2) >> 2;
        if (u0 + u == 0) val = (ld_s16(main0 + 2) + ld_s16(side0 + 2) + 2 * dc + 2) >> 2;
        w |= (uint32_t)val << (16 * e);
      }
      p[h] = w | kBias2;
    }
  }
  if (u0 == 0) {
#pragma unroll
    for (int v = 0; v < 8; v++) {
      if (v0 + v == 0) continue;
      p[4 * v] = set_lo16(p[4 * v], (ld_s16(side0 + 2 * (v0 + v + 1)) + 3 * dc + 2) >> 2);
    }
  }
}
// N = 4 region: four independent PUs (TComPrediction.cpp:755-805, 183-222, 818-841 for N = 4), quadrant-major output
template <class Rec>
CUCD_HD void planar_region16(Rec rec, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const int tr = rec(q, 5), bl = rec(q, 13);
#pragma unroll
    for (int lv = 0; lv < 4; lv++) {
      const int l = rec(q, 9 + lv);
#pragma unroll
      for (int h = 0; h < 2; h++) {
        uint32_t w = 0;
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int lu = 2 * h + e;
          w |= (uint32_t)(((3 - lu) * l + (lu + 1) * tr + (3 - lv) * rec(q, lu + 1) + (lv + 1) * bl + 4) >> 3) << (16 * e);
        }
        p[q * 8 + lv * 2 + h] = w | kBias2;
      }
    }
  }
}
template <class Rec>
CUCD_HD void dc_region16(Rec rec, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    int sum = 4;
#pragma unroll
    for (int i = 1; i <= 4; i++) sum += rec(q, i) + rec(q, 8 + i);
    const int dc = sum >> 3;
#pragma unroll
    for (int lv = 0; lv < 4; lv++)
#pragma unroll
      for (int h = 0; h < 2; h++) {
        uint32_t w = 0;
#pragma unroll
        for (int e = 0; e < 2; e++) {
          const int lu = 2 * h + e;
          int val = dc;
          if (lv == 0) val = lu == 0 ? (rec(q, 1) + rec(q, 9) + 2 * dc + 2) >> 2 : (rec(q, lu + 1) + 3 * dc + 2) >> 2;
          else if (lu == 0) val = (rec(q, 9 + lv) + 3 * dc + 2) >> 2;
          w |= (uint32_t)val << (16 * e);
        }
        p[q * 8 + lv * 2 + h] = w | kBias2;
      }
  }
}

// ---------------------------------------------------------------------------------------------
// prologue: reference arrays of one CTU straight from the reconstruction plane (frame / replay mode), as tc2; phase 1 is
// tc2::tile_load / tile_store with 16-bit samples
// ---------------------------------------------------------------------------------------------
template <int LOG2N>
CUCD_HD void stage_tile16(int tid, int nthreads, const int16_t* rec, int recStride, int W, int H, int ctuX, int ctuY, uint16_t* t) {
  for (int k = tid; k < tc2::kTileThreads; k += nthreads) {
    tc2::TileLoad l;
    tc2::tile_load(k, rec, recStride, W, H, ctuX, ctuY, l);
    tc2::tile_store<Cfg, LOG2N>(k, W, H, ctuX, ctuY, l, t);
  }
}
template <int LOG2N>
CUCD_HD void put_ref16(unsigned char* store, int ctu, int p, int o, int k, int v) {
  const int slot = pu_slot<LOG2N>(ctu, p);
  const uint16_t h = (uint16_t)(0x6400 | v);
  if (LOG2N == 3) *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(ctu, slot, o, 0) + 2 * k) = h;
  else {
    *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(0, slot, o, 0) + 2 * k) = h;
    *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(1, slot, o, 0) + 2 * k) = h;
  }
}
// Phase 2 (tc2::build_unfiltered): unfiltered arrays with HEVC substitution (TComPattern.cpp:314-521) in closed form
template <int LOG2N>
CUCD_HD void build_unfiltered16(int tid, int ctu, int W, int H, int ctuX, int ctuY, int bitDepth, const uint16_t* t, unsigned char* smem) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, TPP = 256 / C::PUS, SPT = 4 * N / TPP, P = C::TILE_PITCH;
  unsigned char* store = smem + C::STORE_OFF;
  const int p = tid / TPP, sub = tid % TPP;
  if (!smem[C::VALID_OFF + ctu * 256 + p]) return;
  int px, py; demorton(p, px, py);
  const int x0 = px * N, y0 = py * N;
  const PuAvail a = pu_avail<LOG2N>(ctuX + x0, ctuY + y0, W, H);
  const uint16_t* rowT = y0 == 0 ? t + C::TILE_TOP + C::TILE_X0 + x0 - 1 : t + (y0 - 1) * P + C::TILE_X0 + x0 - 1;   // rowT[k] = T[k]
  const uint16_t* colL = t + (y0 - 1) * P + C::TILE_X0 + x0 - 1;                                                    // colL[k * P] = L[k], k >= 1
  const int firstAvail = a.lenL > 0 ? colL[a.lenL * P] : (a.availC ? rowT[0] : (a.lenT > 0 ? rowT[1] : (1 << (bitDepth - 1))));
  const int cval = a.availC ? rowT[0] : (a.lenL > 0 ? colL[P] : firstAvail);
  const int tailT = a.lenT > 0 ? rowT[a.lenT] : cval;
  if (LOG2N == 2) {
    // one thread per PU: both records (16 fp16 slots each) leave as two 128-bit stores into the A1 operand
    uint32_t tv[9], lv[9];
    tv[0] = lv[0] = (uint32_t)cval;
#pragma unroll
    for (int k = 1; k <= 8; k++) {
      tv[k] = (uint32_t)(k <= a.lenT ? (int)rowT[k] : tailT);
      lv[k] = (uint32_t)(k <= a.lenL ? (int)colL[k * P] : firstAvail);
    }
    auto w2 = [](uint32_t lo, uint32_t hi) { return lo | (hi << 16) | kBias2; };
    uint32_t* r0a = reinterpret_cast<uint32_t*>(smem + rec_slot_off(ctu, 0, p, 0));   // main = T, side = L
    uint32_t* r0b = reinterpret_cast<uint32_t*>(smem + rec_slot_off(ctu, 0, p, 8));
    uint32_t* r1a = reinterpret_cast<uint32_t*>(smem + rec_slot_off(ctu, 1, p, 0));   // main = L, side = T
    uint32_t* r1b = reinterpret_cast<uint32_t*>(smem + rec_slot_off(ctu, 1, p, 8));
    r0a[0] = w2(tv[0], tv[1]); r0a[1] = w2(tv[2], tv[3]); r0a[2] = w2(tv[4], tv[5]); r0a[3] = w2(tv[6], tv[7]);
    r0b[0] = w2(tv[8], lv[1]); r0b[1] = w2(lv[2], lv[3]); r0b[2] = w2(lv[4], lv[5]); r0b[3] = kConstWord;
    r1a[0] = w2(lv[0], lv[1]); r1a[1] = w2(lv[2], lv[3]); r1a[2] = w2(lv[4], lv[5]); r1a[3] = w2(lv[6], lv[7]);
    r1b[0] = w2(lv[8], tv[1]); r1b[1] = w2(tv[2], tv[3]); r1b[2] = w2(tv[4], tv[5]); r1b[3] = kConstWord;
    return;
  }
  if (sub == 0) { put_ref16<LOG2N>(store, ctu, p, 0, 0, cval); put_ref16<LOG2N>(store, ctu, p, 1, 0, cval); }
  int dcSum = 0, vals[SPT];                          // loads first, stores afterwards (see tc2::build_unfiltered)
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;                     // 0 .. 4N-1
    const int o = j >= 2 * N, k = j - o * 2 * N + 1; // T[k] or L[k]
    if (o == 0) vals[e] = k <= a.lenT ? rowT[k] : tailT;
    else vals[e] = k <= a.lenL ? colL[k * P] : firstAvail;
    if (k <= N) dcSum += vals[e];
  }
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    put_ref16<LOG2N>(store, ctu, p, o, k, vals[e]);
  }
  int* dst = reinterpret_cast<int*>(smem + C::DC_OFF) + ctu * 64 + p;
#if defined(__CUDA_ARCH__)
  if (dcSum) atomicAdd(dst, dcSum);
#else
  *dst += dcSum;
#endif
}
// Phase 3 (tc2::build_filtered): smoothed arrays (TComPattern.cpp:185-283)
template <int LOG2N>
CUCD_HD void build_filtered16(int tid, int ctu, int strongEnabled, int bitDepth, unsigned char* smem) {
  typedef Cfg<LOG2N> C;
  if (!C::HAS_FILT) return;
  constexpr int N = C::N, TPP = 256 / C::PUS, SPT = 4 * N / TPP;
  unsigned char* store = smem + C::STORE_OFF;
  const int p = tid / TPP, sub = tid % TPP;
  if (!smem[C::VALID_OFF + ctu * 256 + p]) return;
  const int slot = pu_slot<LOG2N>(ctu, p);
  const int g0 = LOG2N == 3 ? ctu : 0;
  const unsigned char* T = store + arr_k0_off<LOG2N>(g0, slot, 0, 0);
  const unsigned char* L = store + arr_k0_off<LOG2N>(g0, slot, 1, 0);
  bool strong = false;
  const int tl = ld_s16(T), bl = ld_s16(L + 4 * N), tr = ld_s16(T + 4 * N);
  if (LOG2N == 5 && strongEnabled) {
    const int thr = 1 << (bitDepth - 5);
    strong = iabs32(bl + tl - 2 * ld_s16(L + 2 * N)) < thr && iabs32(tl + tr - 2 * ld_s16(T + 2 * N)) < thr;
  }
  auto put = [&](int o, int k, int v) {
    const uint16_t h = (uint16_t)(0x6400 | v);
    if (LOG2N == 3) *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(ctu, slot, o, 1) + 2 * k) = h;
    else {
      *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(0, slot, o, 1) + 2 * k) = h;
      *reinterpret_cast<uint16_t*>(store + arr_k0_off<LOG2N>(1, slot, o, 1) + 2 * k) = h;
    }
  };
  if (sub == 0) {
    const int c = strong ? tl : (ld_s16(L + 2) + 2 * tl + ld_s16(T + 2) + 2) >> 2;
    put(0, 0, c); put(1, 0, c);
  }
  int vals[SPT];
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    const unsigned char* A = o ? L : T;
    if (k == 2 * N) vals[e] = ld_s16(A + 2 * k);
    else if (strong) vals[e] = o ? (k * bl + (2 * N - k) * tl + N) >> (LOG2N + 1) : ((2 * N - k) * tl + k * tr + N) >> (LOG2N + 1);
    else vals[e] = (ld_s16(A + 2 * (k - 1)) + 2 * ld_s16(A + 2 * k) + ld_s16(A + 2 * (k + 1)) + 2) >> 2;
  }
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    put(o, k, vals[e]);
  }
}
// projected samples of a negative-angle round (tc2::build_ext_group): store[main][-j] = store[side][(128 + j*inv) >> 8],
// two entries per aligned 32-bit store; the fp16 patterns are copied as they are
template <int LOG2N>
CUCD_HD void build_ext_group16(int rowTid, int grp, int inv, int filt, unsigned char* store) {
  typedef Cfg<LOG2N> C;
  constexpr int TPP = LOG2N == 2 ? 1 : 128 / (2 * C::SLOTS);
  constexpr int EPT = C::N / TPP;
  static_assert(LOG2N == 2 || EPT % 2 == 0, "entries are produced two at a time");
  const int pair = rowTid / TPP, sub = rowTid % TPP, slot = pair >> 1, o = pair & 1;
  const int mainOff = arr_k0_off<LOG2N>(grp, slot, o, filt);
  const unsigned char* side = store + arr_k0_off<LOG2N>(grp, slot, o ^ 1, filt);
  int t = 128 + (sub * EPT + 1) * inv;                         // 128 + j * inv of the thread's first entry j
  uint32_t* dst = reinterpret_cast<uint32_t*>(store + mainOff - 2 * (sub * EPT) - 4);   // entries j, j+1 are the high, low half of this word
#pragma unroll
  for (int q = 0; q < EPT / 2; q++) {
    constexpr int kMax = 2 * C::N;
    const uint32_t hi = *reinterpret_cast<const uint16_t*>(side + 2 * imin32(t >> 8, kMax));
    const uint32_t lo = *reinterpret_cast<const uint16_t*>(side + 2 * imin32((t + inv) >> 8, kMax));
    dst[-q] = lo | (hi << 16);
    t += 2 * inv;
  }
}

}  // namespace tc3
}  // namespace cucd
