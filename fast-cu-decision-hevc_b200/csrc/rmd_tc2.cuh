// rmd_tc2.cuh - per-thread logic of the tensor-core RMD frame kernel (8-bit content, sm_100a).
//
// Both the 33 angular PREDICTIONS and the Hadamard SATD run on tcgen05 (kind::i8); the integer ALU only
// moves bytes.  Everything here is `__host__ __device__` like rmd_core.cuh, so tests/emul replays the
// kernel's phases on the CPU with the two tensor-core products replaced by exact integer matmuls.
//
// The arithmetic (reference file:line):
//   angular prediction  TComPrediction.cpp:278-409   pred = ((32-f)*ref[k] + f*ref[k+1] + 16) >> 5
//   projection          TComPrediction.cpp:300-322   ref[k<0] = side[(128 + |k|*invAngle) >> 8]
//   SATD                TComRdCost.cpp:1343-1604
//
// MMA 1 (prediction).  A row of the A operand is the tile's WINDOW of its main reference array: 31
// consecutive u8 samples ref[k0 .. k0+30] and a constant 1.  B holds, for every pixel of the 8x8 tile, the
// two interpolation weights scaled by 8 (8*(32-f) <= 248, 8*f) at the pixel's window slots and the rounding
// term 128 at the constant's slot, so   D = 8 * ((32-f)*a + f*b + 16)   and   pred = byte 1 of D.
// (f == 0: weight 255 and constant 255 give (256*a + (255 - a)) >> 8 = a.)  B depends only on the angle
// and on (tile row offset * angle) mod 32, which takes at most 4 values ("phase class"); the 128 rows of
// one MMA share a phase class by construction of the row map.  For N = 4 a row is an 8x8 REGION of four
// PUs, K = 64 (one 16-byte record per PU: main[0..8], side[1..5], 1) and B is block diagonal with the
// negative-angle projection folded into the weights.
// MMA 2 (Hadamard of the residual).  D = source x -(H8 (x) H8) + prediction x +(H8 (x) H8) (block-diagonal H4 (x) H4 for
// N = 4): the row's source tile sits in shared memory as a static A operand for the whole pass, the 64 predicted bytes
// come from TMEM, and the second product accumulates onto the first.  The epilogue only sums |D|.
#pragma once
#include "rmd_chunk.cuh"

namespace cucd {
namespace tc2 {

constexpr int kThreads = 256;           // 2 row groups of 128 rows (TMEM lanes); two CTAs share an SM
constexpr int kGroups = 2;
constexpr int kAngles = 17;             // am = -8 .. 8;  vertical mode 26 + am, horizontal mode 10 - am (am > -8)
constexpr int kWinTableBytes = kAngles * 4 * 2048;
constexpr int kN4TableBytes = kAngles * 4096;

#if defined(__CUDACC__)
__constant__ int c_angleTab[kAngles] = {-32, -26, -21, -17, -13, -9, -5, -2, 0, 2, 5, 9, 13, 17, 21, 26, 32};
__constant__ int c_invTab[kAngles] = {256, 315, 390, 482, 630, 910, 1638, 4096, 0, 4096, 1638, 910, 630, 482, 390, 315, 256};
#endif
CUCD_HD int angle_of_am(int am) {
#if defined(__CUDA_ARCH__)
  return c_angleTab[am + 8];
#else
  return mode_angle(26 + am);
#endif
}
CUCD_HD int inv_angle_of_am(int am) {
#if defined(__CUDA_ARCH__)
  return c_invTab[am + 8];
#else
  return mode_inv_angle(26 + am);
#endif
}
// byte offset of element (row j, k) of a K-major, no-swizzle UMMA operand with 64 rows (see satd_tc.cuh)
CUCD_HD int umma_off64(int j, int k) { return (k >> 4) * 1024 + (j >> 3) * 128 + (j & 7) * 16 + (k & 15); }

CUCD_HD uint32_t bperm(uint32_t a, uint32_t b, uint32_t sel) {
#if defined(__CUDA_ARCH__)
  return __byte_perm(a, b, sel);
#else
  const uint64_t v = ((uint64_t)b << 32) | a;
  uint32_t r = 0;
  for (int i = 0; i < 4; i++) r |= (uint32_t)((v >> (8 * ((sel >> (4 * i)) & 7))) & 0xffu) << (8 * i);
  return r;
#endif
}
CUCD_HD uint32_t sad_acc(uint32_t d, uint32_t h, uint32_t acc) {
#if defined(__CUDA_ARCH__)
  return __sad((int)d, (int)h, acc);
#else
  const int v = (int)d - (int)h;
  return acc + (uint32_t)(v < 0 ? -v : v);
#endif
}

// ---------------------------------------------------------------------------------------------
// window geometry shared by the table generator and the gather
// ---------------------------------------------------------------------------------------------
// lowest local row shift of an 8-row tile: 0 for angle >= 0, (frac0 + 8*angle) >> 5 otherwise
CUCD_HD int win_lmin(int angle, int frac0) { return angle >= 0 ? 0 : ((frac0 + 8 * angle) >> 5); }
// first reference index of the window of the tile at (u0, v0) (orientation coordinates)
CUCD_HD int win_k0(int angle, int u0, int v0) {
  const int t = v0 * angle;
  return u0 + (t >> 5) + 1 + win_lmin(angle, t & 31);
}

// B operand of MMA 1 for N >= 8: table[(am + 8) * 4 + fc] = 64 pixels x 32 slots, UMMA layout, 2 KB each
inline void fill_win_tables(uint8_t* dst /*kWinTableBytes*/) {
  for (int i = 0; i < kWinTableBytes; i++) dst[i] = 0;
  for (int am = -8; am <= 8; am++)
    for (int fc = 0; fc < 4; fc++) {
      uint8_t* t = dst + ((am + 8) * 4 + fc) * 2048;
      const int a = angle_of_am(am), frac0 = fc * 8, lmin = win_lmin(a, frac0);
      for (int v = 0; v < 8; v++) {
        const int d = frac0 + (v + 1) * a, li = d >> 5, f = d & 31;
        for (int u = 0; u < 8; u++) {
          const int j = v * 8 + u, s = u + li - lmin;
          if (f == 0) { t[umma_off64(j, s)] = 255; t[umma_off64(j, 31)] = 255; }
          else { t[umma_off64(j, s)] = (uint8_t)(8 * (32 - f)); t[umma_off64(j, s + 1)] = (uint8_t)(8 * f); t[umma_off64(j, 31)] = 128; }
        }
      }
    }
}
// slot of reference sample k inside a PU record of the N = 4 path: main[0..8] at 0..8, side[1..5] at 9..13, 1 at 15
CUCD_HD int n4_slot(int k, int inv) { return k >= 0 ? k : 8 + ((128 - k * inv) >> 8); }
// B operand of MMA 1 for N = 4: table[am + 8] = 64 region pixels x 64 slots (4 records), 4 KB each
inline void fill_n4_tables(uint8_t* dst /*kN4TableBytes*/) {
  for (int i = 0; i < kN4TableBytes; i++) dst[i] = 0;
  for (int am = -8; am <= 8; am++) {
    uint8_t* t = dst + (am + 8) * 4096;
    const int a = angle_of_am(am), inv = inv_angle_of_am(am);
    for (int v = 0; v < 8; v++)
      for (int u = 0; u < 8; u++) {
        const int j = v * 8 + u, q = (v >> 2) * 2 + (u >> 2), lv = v & 3, lu = u & 3;
        const int d = (lv + 1) * a, f = d & 31, k = lu + (d >> 5) + 1;
        if (f == 0) { t[umma_off64(j, q * 16 + n4_slot(k, inv))] = 255; t[umma_off64(j, q * 16 + 15)] = 255; }
        else {
          t[umma_off64(j, q * 16 + n4_slot(k, inv))] = (uint8_t)(8 * (32 - f));
          t[umma_off64(j, q * 16 + n4_slot(k + 1, inv))] = (uint8_t)(8 * f);
          t[umma_off64(j, q * 16 + 15)] = 128;
        }
      }
  }
}

// ---------------------------------------------------------------------------------------------
// shared memory of the CTA
// ---------------------------------------------------------------------------------------------
// u8 reference arrays of the N >= 8 path: element k of an array lives at byte  arr + N + k,  k = -N .. 2N + 20
// ([-N, -1] holds the projected samples of the negative-angle mode being evaluated, TComPrediction.cpp:300-322).
// Arrays of one PU: index (filt * 2 + o), o = 0: main = above row ("T"), o = 1: main = left column ("L").
// Each of the two row groups owns a PRIVATE copy of the arrays of the PUs its rows touch ("slots"), so that the
// projected part can be rewritten per mode round with row-group barriers only (the groups run unsynchronised).
//
// Work of one CTA: N = 4, 8: two CTUs, row group = CTU;  N = 16: two CTUs, row group = phase class (tile row
// parity);  N = 32, 64: four CTUs in two passes, pass p evaluates the phase classes {2p, 2p+1}.
template <int LOG2N>
struct Cfg {
  typedef Geo<LOG2N> G;
  static constexpr int al16(int v) { return (v + 15) & ~15; }
  static constexpr int N = 1 << LOG2N;
  static constexpr int PUS = 4096 / (N * N);                     // PUs of one CTU at this depth
  static constexpr int CTUS = LOG2N >= 5 ? 4 : 2;                // CTUs per CTA
  static constexpr int PASSES = LOG2N >= 5 ? 2 : 1;
  static constexpr bool HAS_FILT = LOG2N >= 3 && LOG2N <= 5;
  static constexpr int NARR = HAS_FILT ? 4 : 2;
  static constexpr int AS8 = (3 * N + 21 + 3) & ~3;
  static constexpr int PU_RAW = NARR * AS8;
  // odd number of words: lanes of different PUs hit different banks.  N = 64: a warp reads one PU, and the 432 bytes of a CTU's slot stay a
  // 16-byte multiple, as its bulk copy needs (border pre-pass, rmd_tc_frame.cuh)
  static constexpr int PU_BYTES = LOG2N == 6 ? PU_RAW : PU_RAW + (((PU_RAW >> 2) & 1) ? 0 : 4);
  static constexpr int SLOTS = LOG2N == 3 ? 64 : CTUS * PUS;     // PUs seen by one row group
  static constexpr int GROUP_BYTES = LOG2N == 2 ? 0 : al16(16 + SLOTS * PU_BYTES);
  static constexpr int STORE_BYTES = LOG2N == 2 ? CTUS * 256 * 2 * 16 : kGroups * GROUP_BYTES;   // N = 4: shared 16-byte records [ctu][o][pu]
  static constexpr int B1_BYTES = LOG2N == 2 ? 4096 : 2048;      // one MMA 1 weight operand
  static constexpr int ACC_ELEM = LOG2N == 2 ? 2 : 4;            // costs are staged in shared memory: uint32, N = 4: uint16 (<= 8160 for 8-bit content)
  static constexpr bool EDGE = LOG2N <= 4;                       // luma edge filters (DC, pure vertical / horizontal)
  // byte offsets inside dynamic shared memory
  static constexpr int HAD_OFF = 0;                              // +H at 0, -H at 4096 (B operands of MMA 2)
  static constexpr int B1_OFF = HAD_OFF + 8192;                  // [group][buffer]
  static constexpr int A1_OFF = B1_OFF + kGroups * 2 * B1_BYTES; // [group]: two 4 KB window operands (N >= 8) or one static 8 KB record operand (N = 4)
  static constexpr int AORG_OFF = A1_OFF + kGroups * 8192;       // [group]: the rows' SOURCE tiles as a 128 x 64-byte operand: MMA 2 accumulates -H x source
  static constexpr int BAR_OFF = AORG_OFF + kGroups * 8192;
  static constexpr int VALID_OFF = BAR_OFF + 128;
  static constexpr int DC_OFF = VALID_OFF + CTUS * 256;          // int32 [ctu][64]: sum of the N above + N left samples (N >= 8)
  static constexpr int STORE_OFF = DC_OFF + CTUS * 64 * 4;
  static constexpr int ACC_OFF = STORE_OFF + al16(STORE_BYTES);
  static constexpr int TOTAL = ACC_OFF + al16(CTUS * PUS * kNumModes * ACC_ELEM);
  // u8 copy of the reconstruction around each CTU while the reference arrays are built (frame mode): the border pre-pass holds one
  // per CTA; the CPU replay of the in-kernel prologue (tests/emul/rmd_tc2_emul.cpp) stages them at TILE_OFF, in the MMA 1 operand
  // buffers, which are first written after the prologue
  static constexpr int TILE_OFF = B1_OFF;
  static constexpr int TILE_PITCH = 68;                          // 17 words: a column walk touches 32 different banks
  static constexpr int TILE_X0 = 4;                              // tile[y][x] = t[y * TILE_PITCH + TILE_X0 + x], x = -1 .. 63
  static constexpr int TILE_TOP = 64 * TILE_PITCH;               // row y = -1: top[x] = t[TILE_TOP + TILE_X0 + x], x = -1 .. 127
  static constexpr int TILE_BYTES = al16(TILE_TOP + 136);
  static_assert(CTUS * TILE_BYTES <= kGroups * 2 * B1_BYTES + kGroups * 8192, "tiles must fit the aliased operand buffers");
};
constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int kSmemBytes = cmax(cmax(cmax(Cfg<2>::TOTAL, Cfg<3>::TOTAL), cmax(Cfg<4>::TOTAL, Cfg<5>::TOTAL)), Cfg<6>::TOTAL);

// slot of PU (ctu, pu) inside the private store of the row groups that use it
template <int LOG2N> CUCD_HD int pu_slot2(int ctu, int pu) { return LOG2N == 3 ? pu : ctu * Cfg<LOG2N>::PUS + pu; }
// byte offset (from the start of the store) of element k = 0 of array (slot, o, filt) in row group `grp`'s copy
template <int LOG2N> CUCD_HD int arr_k0_off(int grp, int slot, int o, int filt) {
  typedef Cfg<LOG2N> C;
  return grp * C::GROUP_BYTES + 16 + slot * C::PU_BYTES + (filt * 2 + o) * C::AS8 + C::N;
}
CUCD_HD int rec_off(int ctu, int o, int pu) { return ((ctu * 2 + o) * 256 + pu) * 16; }

// Frame mode: the border pre-pass (rmd_border_prep_kernel) builds the reference arrays of every CTU at every depth once, as an
// IMAGE per (CTU, depth): the bytes the prologue of the CTU's CTA would write into one row-group copy of the store - N = 4: the
// records [o][pu], N = 8: the slots of the CTU's row group, N >= 16: the CTU's PUS consecutive slots - then its DC sums (N >= 8).
// Both parts are 16-byte multiples; the RMD CTA places them with cp.async.bulk.  The images of a CTU are consecutive, depth 0 (N = 64)
// first: kPrepCtuBytes per CTU.
template <int LOG2N>
struct PrepSize {
  typedef Cfg<LOG2N> C;
  static constexpr int STORE = LOG2N == 2 ? 2 * 256 * 16 : C::PUS * C::PU_BYTES;
  static constexpr int DC = LOG2N == 2 ? 0 : C::al16(C::PUS * 4);
  static constexpr int BYTES = STORE + DC;
  static_assert(STORE % 16 == 0, "a bulk copy moves 16-byte multiples");
};
constexpr int kPrepCtuBytes = PrepSize<2>::BYTES + PrepSize<3>::BYTES + PrepSize<4>::BYTES + PrepSize<5>::BYTES + PrepSize<6>::BYTES;
template <int LOG2N> CUCD_HD constexpr int prep_off() {
  return (LOG2N < 6 ? PrepSize<6>::BYTES : 0) + (LOG2N < 5 ? PrepSize<5>::BYTES : 0) + (LOG2N < 4 ? PrepSize<4>::BYTES : 0) + (LOG2N < 3 ? PrepSize<3>::BYTES : 0);
}
// where the store image of the CTA's CTU c lands in row group grp's copy of the store (N <= 8: one copy, grp unused)
template <int LOG2N> CUCD_HD int prep_store_off(int grp, int c) {
  typedef Cfg<LOG2N> C;
  return LOG2N == 2 ? rec_off(c, 0, 0) : (LOG2N == 3 ? c * C::GROUP_BYTES + 16 : grp * C::GROUP_BYTES + 16 + c * C::PUS * C::PU_BYTES);
}
// The bulk copies that place the image of the CTA's CTU c: one per row-group copy of the store (N >= 16: two) and the DC sums.
// Copy i: `bytes` bytes from offset `src` of the image to offset `dst` of the CTA's shared memory.
struct PrepCopy { int dst, src, bytes; };
template <int LOG2N> CUCD_HD constexpr int prep_copies() { return LOG2N == 2 ? 1 : (LOG2N == 3 ? 2 : 3); }
template <int LOG2N> CUCD_HD PrepCopy prep_copy(int c, int i) {
  typedef Cfg<LOG2N> C;
  typedef PrepSize<LOG2N> S;
  if (LOG2N >= 3 && i == prep_copies<LOG2N>() - 1) return PrepCopy{C::DC_OFF + c * 256, S::STORE, S::DC};
  return PrepCopy{C::STORE_OFF + prep_store_off<LOG2N>(i, c), 0, S::STORE};
}
// bytes of the copies of one CTU (what the CTA's mbarrier expects per CTU)
template <int LOG2N> CUCD_HD constexpr int prep_copy_bytes() { return (prep_copies<LOG2N>() - (LOG2N >= 3 ? 1 : 0)) * PrepSize<LOG2N>::STORE + PrepSize<LOG2N>::DC; }
// the cost of element i (= pu * 35 + mode) of the CTA's CTU c in the accumulators at ACC_OFF: uint16 for N = 4, uint32 otherwise
template <int LOG2N> struct CostRead {
  const uint32_t* acc;
  CUCD_HD uint32_t operator()(int c, int i) const {
    const int e = c * Cfg<LOG2N>::PUS * kNumModes + i;
    return LOG2N == 2 ? (uint32_t)reinterpret_cast<const uint16_t*>(acc)[e] : acc[e];
  }
};

// ---------------------------------------------------------------------------------------------
// which tile a thread (= MMA row = TMEM lane) owns
// ---------------------------------------------------------------------------------------------
struct Row {
  int ctu;      // inside the CTA
  int o;        // 0: true orientation (planar + modes 18..34), 1: transposed (DC + modes 2..17)
  int pu;       // CTU-local PU (z order); N = 4: the REGION index, its PUs are 4*pu .. 4*pu+3
  int u0, v0;   // tile origin inside the PU in orientation coordinates (u along the main reference)
};
template <int LOG2N> struct RowSeg { static constexpr int value = LOG2N <= 3 ? 1 : (LOG2N == 4 ? 2 : (LOG2N == 5 ? 4 : 16)); };   // lanes sharing (PU, orientation)
template <int LOG2N>
CUCD_HD Row row_map(int tid, int pass) {
  const int g = tid >> 7, wq = (tid >> 5) & 3, lane = tid & 31;
  Row r;
  if (LOG2N <= 3) { r.ctu = g; r.o = wq >> 1; r.pu = (wq & 1) * 32 + lane; r.u0 = 0; r.v0 = 0; }
  else if (LOG2N == 4) { r.ctu = wq >> 1; r.o = wq & 1; r.pu = lane >> 1; r.u0 = 8 * (lane & 1); r.v0 = 8 * g; }
  else if (LOG2N == 5) { r.ctu = wq; r.o = lane >> 4; r.pu = (lane >> 2) & 3; r.u0 = 8 * (lane & 3); r.v0 = 8 * (2 * pass + g); }
  else { r.ctu = wq; r.o = lane >> 4; r.pu = 0; r.u0 = 8 * (lane & 7); r.v0 = 8 * (2 * pass + g + 4 * ((lane >> 3) & 1)); }
  return r;
}
// phase class of a row group: (v0 / 8) mod 4 is the same for its 128 rows
template <int LOG2N>
CUCD_HD int group_frac0(int grp, int pass, int angle) {
  const int t = LOG2N <= 3 ? 0 : (LOG2N == 4 ? grp : 2 * pass + grp);
  return (8 * t * angle) & 31;
}

// ---------------------------------------------------------------------------------------------
// byte tiles
// ---------------------------------------------------------------------------------------------
// w[16]: word 2*y + h = pixels (y, 4h .. 4h+3).  Transpose the whole 8x8 (blocks = true) or each 4x4 quadrant in place.
CUCD_HD void transpose4x4_bytes(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t* o) {
  const uint32_t t0 = bperm(a0, a1, 0x5140), t1 = bperm(a2, a3, 0x5140);   // (a0.0 a1.0 a0.1 a1.1), (a2.0 a3.0 a2.1 a3.1)
  const uint32_t t2 = bperm(a0, a1, 0x7362), t3 = bperm(a2, a3, 0x7362);   // (a0.2 a1.2 a0.3 a1.3), ...
  o[0] = bperm(t0, t1, 0x5410); o[1] = bperm(t0, t1, 0x7632);
  o[2] = bperm(t2, t3, 0x5410); o[3] = bperm(t2, t3, 0x7632);
}
CUCD_HD void tile_transpose_bytes(const uint32_t* w, uint32_t* d, bool whole) {
#pragma unroll
  for (int qy = 0; qy < 2; qy++)
#pragma unroll
    for (int qx = 0; qx < 2; qx++) {
      uint32_t o[4];
      transpose4x4_bytes(w[(qy * 4 + 0) * 2 + qx], w[(qy * 4 + 1) * 2 + qx], w[(qy * 4 + 2) * 2 + qx], w[(qy * 4 + 3) * 2 + qx], o);
      const int dy = whole ? qx : qy, dx = whole ? qy : qx;
#pragma unroll
      for (int i = 0; i < 4; i++) d[(dy * 4 + i) * 2 + dx] = o[i];
    }
}

// ---------------------------------------------------------------------------------------------
// MMA 1 operand of a row (N >= 8): 32 bytes starting at byte address q of the store, last byte := 1
// ---------------------------------------------------------------------------------------------
CUCD_HD void gather_window(const unsigned char* store, int q, uint32_t* w8) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(store + (q & ~3));
  const uint32_t sel = 0x3210u + 0x1111u * (uint32_t)(q & 3);
  uint32_t x[9];
#pragma unroll
  for (int j = 0; j < 9; j++) x[j] = s[j];
#pragma unroll
  for (int j = 0; j < 8; j++) w8[j] = bperm(x[j], x[j + 1], sel);
  w8[7] = (w8[7] & 0x00ffffffu) | 0x01000000u;
}
// epilogue 1: packed[j] = (D[2j] & 0xffff) | (D[2j+1] << 16)  ->  4 predicted pixels per word
CUCD_HD void pack_pred(const uint32_t* packed /*2 * NW*/, uint32_t* out /*NW*/, int nw) {
#pragma unroll
  for (int i = 0; i < 8; i++) if (i < nw) out[i] = bperm(packed[2 * i], packed[2 * i + 1], 0x7531);
}
CUCD_HD int clip8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

// pure vertical / horizontal modes, N <= 16: first column gets the edge filter (TComPrediction.cpp:346-363)
// main/side: element 0 = corner.  p = 16 words of the tile, v0 = first tile row inside the PU.
CUCD_HD void patch_edge0_tile(const unsigned char* main0, const unsigned char* side0, int v0, uint32_t* p) {
  const int m1 = main0[1], s0 = side0[0];
#pragma unroll
  for (int v = 0; v < 8; v++) {
    const int val = clip8(m1 + (((int)side0[v0 + v + 1] - s0) >> 1));
    p[2 * v] = (p[2 * v] & 0xffffff00u) | (uint32_t)val;
  }
}
CUCD_HD void patch_edge0_region4(const unsigned char* rec /*4 records*/, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const unsigned char* r = rec + q * 16;
    const int m1 = r[1], s0 = r[0];
#pragma unroll
    for (int lv = 0; lv < 4; lv++) {
      const int val = clip8(m1 + (((int)r[9 + lv] - s0) >> 1));
      const int w = 2 * ((q >> 1) * 4 + lv) + (q & 1);
      p[w] = (p[w] & 0xffffff00u) | (uint32_t)val;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// planar and DC on the integer ALU (2 of the 35 modes), bytes out.  main/side: element 0 = corner.
// ---------------------------------------------------------------------------------------------
// TComPrediction.cpp:755-805 for the 8x8 tile at (u0, v0) of an N x N PU
// Two pixels per integer: every (hor + vert + N) < 2^15, so pairs live in the 16-bit halves of a word and row /
// column increments (possibly negative) are single integer adds of (stepHi << 16) + stepLo.
CUCD_HD void planar_tile(int log2n, const unsigned char* T, const unsigned char* L, int u0, int v0, uint32_t* p) {
  const int N = 1 << log2n;
  const int tr = T[N + 1], bl = L[N + 1];
  uint32_t V[4], VS[4];                              // vert term of columns (2j, 2j+1) at row v0, and its per-row step
#pragma unroll
  for (int j = 0; j < 4; j++) {
    const int t0 = T[u0 + 2 * j + 1], t1 = T[u0 + 2 * j + 2];
    V[j] = (uint32_t)((N - 1 - v0) * t0 + (v0 + 1) * bl) + ((uint32_t)((N - 1 - v0) * t1 + (v0 + 1) * bl) << 16);
    VS[j] = (uint32_t)(bl - t0) + ((uint32_t)(bl - t1) << 16);
  }
  const uint32_t mask = 0x00ff00ffu;
#pragma unroll
  for (int v = 0; v < 8; v++) {
    const int l = L[v0 + v + 1], hs = tr - l;
    const int b = (N - 1 - u0) * l + (u0 + 1) * tr + N;      // hor term + rounding at column u0
    uint32_t H = (uint32_t)b + ((uint32_t)(b + hs) << 16);
    const uint32_t H2 = (uint32_t)(2 * hs) * 0x00010001u;
    uint32_t q[4];
#pragma unroll
    for (int j = 0; j < 4; j++) { q[j] = ((H + V[j]) >> (log2n + 1)) & mask; H += H2; V[j] += VS[j]; }
    p[2 * v] = bperm(q[0], q[1], 0x6420); p[2 * v + 1] = bperm(q[2], q[3], 0x6420);
  }
}
// TComPrediction.cpp:183-222, 818-841
CUCD_HD void dc_tile(int dc, bool edge, const unsigned char* main0, const unsigned char* side0, int u0, int v0, uint32_t* p) {
  const uint32_t dc4 = (uint32_t)dc * 0x01010101u;
#pragma unroll
  for (int i = 0; i < 16; i++) p[i] = dc4;
  if (!edge) return;
  if (v0 == 0) {
    uint32_t w0 = 0, w1 = 0;
#pragma unroll
    for (int u = 0; u < 8; u++) {
      int val = ((int)main0[u0 + u + 1] + 3 * dc + 2) >> 2;
      if (u0 + u == 0) val = ((int)main0[1] + (int)side0[1] + 2 * dc + 2) >> 2;
      if (u < 4) w0 |= (uint32_t)val << (8 * u); else w1 |= (uint32_t)val << (8 * (u - 4));
    }
    p[0] = w0; p[1] = w1;
  }
  if (u0 == 0) {
#pragma unroll
    for (int v = 0; v < 8; v++) {
      if (v0 + v == 0) continue;
      const int val = ((int)side0[v0 + v + 1] + 3 * dc + 2) >> 2;
      p[2 * v] = (p[2 * v] & 0xffffff00u) | (uint32_t)val;
    }
  }
}
// N = 4 region: four independent PUs, records [main 0..8 | side 1..5 | 0 | 1]
CUCD_HD void planar_region4(const unsigned char* rec, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const unsigned char* r = rec + q * 16;
    const int tr = r[5], bl = r[13];
#pragma unroll
    for (int lv = 0; lv < 4; lv++) {
      const int l = r[9 + lv];
      uint32_t w = 0;
#pragma unroll
      for (int lu = 0; lu < 4; lu++) {
        const int val = ((3 - lu) * l + (lu + 1) * tr + (3 - lv) * (int)r[lu + 1] + (lv + 1) * bl + 4) >> 3;
        w |= (uint32_t)val << (8 * lu);
      }
      p[2 * ((q >> 1) * 4 + lv) + (q & 1)] = w;
    }
  }
}
CUCD_HD void dc_region4(const unsigned char* rec, uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 4; q++) {
    const unsigned char* r = rec + q * 16;
    int sum = 4;
#pragma unroll
    for (int i = 1; i <= 4; i++) sum += (int)r[i] + (int)r[8 + i];
    const int dc = sum >> 3;
#pragma unroll
    for (int lv = 0; lv < 4; lv++) {
      uint32_t w = (uint32_t)dc * 0x01010101u;
      if (lv == 0) {
        w = 0;
#pragma unroll
        for (int lu = 0; lu < 4; lu++) {
          int val = ((int)r[lu + 1] + 3 * dc + 2) >> 2;
          if (lu == 0) val = ((int)r[1] + (int)r[9] + 2 * dc + 2) >> 2;
          w |= (uint32_t)val << (8 * lu);
        }
      } else {
        w = (w & 0xffffff00u) | (uint32_t)(((int)r[9 + lv] + 3 * dc + 2) >> 2);
      }
      p[2 * ((q >> 1) * 4 + lv) + (q & 1)] = w;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// prologue: reference arrays of one CTU straight from the reconstruction plane (frame / replay mode)
// ---------------------------------------------------------------------------------------------
// 8 samples = one 128-bit load (g++ builds the emulators without the CUDA headers, so no uint4), and half of it
struct alignas(16) Vec16 { uint32_t x, y, z, w; };
struct alignas(8) Vec8 { uint32_t x, y; };

// Phase 1 (frame / replay mode): the CTU's 64x64 reconstruction block, the row above it (x = -1 .. 127) and the column left of it, split
// into the global loads (tile_load), issued for all the CTA's CTUs before anything waits, and the shared-memory stores (tile_store).
// A thread of the CTA's 256 holds two 8-sample chunks of the block, thread t < 64 the left neighbour of row t, thread t < 129 the
// above neighbour x = t - 1.  Samples outside the picture are not stored (never consumed: availability masks them).
// Shared with tc3 (uint16 tiles); the frame kernels' set-up is rmd_tc_frame.cuh setup_loads.
constexpr int kTileThreads = 256;
struct TileLoad { Vec16 v[2]; int left, top; };
CUCD_HD void tile_load(int tid, const int16_t* rec, int recStride, int W, int H, int ctuX, int ctuY, TileLoad& t) {
#pragma unroll
  for (int it = 0; it < 2; it++) {
    const int idx = tid + it * kTileThreads, y = idx >> 3, x = (idx & 7) * 8;
    t.v[it] = Vec16{0u, 0u, 0u, 0u};
    if (ctuY + y < H && ctuX + x < W) t.v[it] = *reinterpret_cast<const Vec16*>(rec + (size_t)(ctuY + y) * recStride + ctuX + x);
  }
  t.left = 0; t.top = 0;
  if (ctuX > 0 && tid < 64 && ctuY + tid < H) t.left = rec[(size_t)(ctuY + tid) * recStride + ctuX - 1];
  const int gx = ctuX - 1 + tid;
  if (ctuY > 0 && tid < 129 && gx >= 0 && gx < W) t.top = rec[(size_t)(ctuY - 1) * recStride + gx];
}
// tile[y][x] = dst[y * TILE_PITCH + TILE_X0 + x], top[x] = dst[TILE_TOP + TILE_X0 + x]: bytes (the low byte of each sample, tc2) or
// the samples themselves (uint16, tc3)
template <template <int> class Cfg, int LOG2N, class T>
CUCD_HD void tile_store(int tid, int W, int H, int ctuX, int ctuY, const TileLoad& t, T* dst) {
  typedef Cfg<LOG2N> C;
#pragma unroll
  for (int it = 0; it < 2; it++) {
    const int idx = tid + it * kTileThreads, y = idx >> 3, x = (idx & 7) * 8;
    if (ctuY + y >= H || ctuX + x >= W) continue;
    const Vec16& v = t.v[it];
    if (sizeof(T) == 1) {
      uint32_t* d = reinterpret_cast<uint32_t*>(dst + y * C::TILE_PITCH + C::TILE_X0 + x);
      d[0] = bperm(v.x, v.y, 0x6420); d[1] = bperm(v.z, v.w, 0x6420);
    } else {
      Vec8* d = reinterpret_cast<Vec8*>(dst + y * C::TILE_PITCH + C::TILE_X0 + x);      // rows are 8-byte aligned
      d[0] = Vec8{v.x, v.y}; d[1] = Vec8{v.z, v.w};
    }
  }
  if (ctuX > 0 && tid < 64 && ctuY + tid < H) dst[tid * C::TILE_PITCH + C::TILE_X0 - 1] = (T)t.left;
  const int gx = ctuX - 1 + tid;
  if (ctuY > 0 && tid < 129 && gx >= 0 && gx < W) dst[C::TILE_TOP + C::TILE_X0 - 1 + tid] = (T)t.top;
}
// phase 1 of one CTU in one call, thread ids tid, tid + nthreads, ... of the 256 (the CPU replay's form)
template <int LOG2N>
CUCD_HD void stage_tile(int tid, int nthreads, const int16_t* rec, int recStride, int W, int H, int ctuX, int ctuY, unsigned char* t) {
  for (int k = tid; k < kTileThreads; k += nthreads) {
    TileLoad l;
    tile_load(k, rec, recStride, W, H, ctuX, ctuY, l);
    tile_store<Cfg, LOG2N>(k, W, H, ctuX, ctuY, l, t);
  }
}

// Phase 2: unfiltered reference arrays with HEVC substitution (TComPattern.cpp:314-521) in closed form.  In
// replay mode availability is positional (z-scan order, TComPattern.cpp:550-727): the left column, the corner
// and the above row are each available or not as a whole, the below-left / above-right extensions are available
// for their first cntBL / cntAR 4-sample units (the neighbouring block precedes the PU in z order; the picture
// edge cuts the run).  Scan order of the substitution: L[2N] .. L[1], corner, T[1] .. T[2N]:
//   a leading unavailable run takes the first available sample, any other unavailable sample its predecessor.
struct PuAvail { int lenL, lenT, availC; };
template <int LOG2N>
CUCD_HD PuAvail pu_avail(int X0, int Y0, int W, int H) {
  constexpr int N = 1 << LOG2N;
  PuAvail a;
  const bool availL = X0 > 0, availA = Y0 > 0;
  int cntBL = 0, cntAR = 0;
  if (availL && unit_available(X0, Y0, X0 - 1, Y0 + N, W, H)) cntBL = imin32(N / 4, (H - (Y0 + N)) >> 2);
  if (availA && unit_available(X0, Y0, X0 + N, Y0 - 1, W, H)) cntAR = imin32(N / 4, (W - (X0 + N)) >> 2);
  a.lenL = availL ? N + 4 * cntBL : 0;
  a.lenT = availA ? N + 4 * cntAR : 0;
  a.availC = availL && availA;
  return a;
}
// write one unfiltered sample (array o: 0 = T, 1 = L; element k) of PU (ctu, p) into the store
template <int LOG2N>
CUCD_HD void put_ref(unsigned char* store, int ctu, int p, int o, int k, int v) {
  if (LOG2N == 2) {
    if (k <= 8) store[rec_off(ctu, o, p) + k] = (unsigned char)v;                   // main of orientation o
    if (k >= 1 && k <= 5) store[rec_off(ctu, o ^ 1, p) + 8 + k] = (unsigned char)v; // side of the other orientation
  } else {
    const int slot = pu_slot2<LOG2N>(ctu, p);
    if (LOG2N == 3) store[arr_k0_off<LOG2N>(ctu, slot, o, 0) + k] = (unsigned char)v;
    else { store[arr_k0_off<LOG2N>(0, slot, o, 0) + k] = (unsigned char)v; store[arr_k0_off<LOG2N>(1, slot, o, 0) + k] = (unsigned char)v; }
  }
}
// 256 / PUS threads share a PU; each produces 4N / (256 / PUS) consecutive samples of the sequence T[1..2N], L[1..2N]
// (N = 4: one thread per PU, 16 samples) and the first of them the corner.
// The `_at` builders write through `prol`, the CTA's shared memory from VALID_OFF on (PU states, DC sums, store: offsets ProlOff), so
// that the border pre-pass can run them on a staging area of that layout (rmd_tc_frame.cuh prep_phase); build_unfiltered /
// build_filtered take the CTA's shared memory itself.
template <int LOG2N> struct ProlOff {
  static constexpr int DC = Cfg<LOG2N>::DC_OFF - Cfg<LOG2N>::VALID_OFF, STORE = Cfg<LOG2N>::STORE_OFF - Cfg<LOG2N>::VALID_OFF;
};
template <int LOG2N>
CUCD_HD void build_unfiltered_at(int tid, int ctu, int W, int H, int ctuX, int ctuY, const unsigned char* t, unsigned char* prol) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, TPP = 256 / C::PUS, SPT = 4 * N / TPP;
  unsigned char* store = prol + ProlOff<LOG2N>::STORE;
  const int p = tid / TPP, sub = tid % TPP;
  if (!prol[ctu * 256 + p]) return;
  int px, py; demorton(p, px, py);
  const int x0 = px * N, y0 = py * N;
  const PuAvail a = pu_avail<LOG2N>(ctuX + x0, ctuY + y0, W, H);
  const unsigned char* rowT = y0 == 0 ? t + C::TILE_TOP + C::TILE_X0 + x0 - 1 : t + (y0 - 1) * C::TILE_PITCH + C::TILE_X0 + x0 - 1;   // rowT[k] = T[k]
  const unsigned char* colL = t + (y0 - 1) * C::TILE_PITCH + C::TILE_X0 + x0 - 1;                                                    // colL[k * PITCH] = L[k], k >= 1
  const int firstAvail = a.lenL > 0 ? colL[a.lenL * C::TILE_PITCH] : (a.availC ? rowT[0] : (a.lenT > 0 ? rowT[1] : 128));
  const int cval = a.availC ? rowT[0] : (a.lenL > 0 ? colL[C::TILE_PITCH] : firstAvail);
  const int tailT = a.lenT > 0 ? rowT[a.lenT] : cval;
  if (LOG2N == 2) {
    // one thread per PU: both 16-byte records are assembled in registers and leave as two 128-bit stores
    uint32_t tv[9], lv[9];
    tv[0] = lv[0] = (uint32_t)cval;
#pragma unroll
    for (int k = 1; k <= 8; k++) {
      tv[k] = (uint32_t)(k <= a.lenT ? (int)rowT[k] : tailT);
      lv[k] = (uint32_t)(k <= a.lenL ? (int)colL[k * C::TILE_PITCH] : firstAvail);
    }
    auto w4 = [](uint32_t b0, uint32_t b1, uint32_t b2, uint32_t b3) { return b0 | (b1 << 8) | (b2 << 16) | (b3 << 24); };
    uint32_t* r0 = reinterpret_cast<uint32_t*>(store + rec_off(ctu, 0, p));       // main = T, side = L
    uint32_t* r1 = reinterpret_cast<uint32_t*>(store + rec_off(ctu, 1, p));       // main = L, side = T
    r0[0] = w4(tv[0], tv[1], tv[2], tv[3]); r0[1] = w4(tv[4], tv[5], tv[6], tv[7]); r0[2] = w4(tv[8], lv[1], lv[2], lv[3]); r0[3] = w4(lv[4], lv[5], 0u, 1u);
    r1[0] = w4(lv[0], lv[1], lv[2], lv[3]); r1[1] = w4(lv[4], lv[5], lv[6], lv[7]); r1[2] = w4(lv[8], tv[1], tv[2], tv[3]); r1[3] = w4(tv[4], tv[5], 0u, 1u);
    return;
  }
  if (sub == 0) {
    put_ref<LOG2N>(store, ctu, p, 0, 0, cval); put_ref<LOG2N>(store, ctu, p, 1, 0, cval);
    if (LOG2N == 2) { store[rec_off(ctu, 0, p) + 14] = 0; store[rec_off(ctu, 0, p) + 15] = 1; store[rec_off(ctu, 1, p) + 14] = 0; store[rec_off(ctu, 1, p) + 15] = 1; }
  }
  // all the samples are read before the first one is stored: the stores may alias the tile as far as the compiler can tell, and
  // interleaved they would serialise every shared-memory round trip
  int dcSum = 0, vals[SPT];
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;                     // 0 .. 4N-1
    const int o = j >= 2 * N, k = j - o * 2 * N + 1; // T[k] or L[k]
    if (o == 0) vals[e] = k <= a.lenT ? rowT[k] : tailT;
    else vals[e] = k <= a.lenL ? colL[k * C::TILE_PITCH] : firstAvail;
    if (k <= N) dcSum += vals[e];
  }
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    put_ref<LOG2N>(store, ctu, p, o, k, vals[e]);
  }
  if (LOG2N >= 3) {
    int* dst = reinterpret_cast<int*>(prol + ProlOff<LOG2N>::DC) + ctu * 64 + p;
#if defined(__CUDA_ARCH__)
    if (dcSum) atomicAdd(dst, dcSum);
#else
    *dst += dcSum;
#endif
  }
}
template <int LOG2N>
CUCD_HD void build_unfiltered(int tid, int ctu, int W, int H, int ctuX, int ctuY, const unsigned char* t, unsigned char* smem) {
  build_unfiltered_at<LOG2N>(tid, ctu, W, H, ctuX, ctuY, t, smem + Cfg<LOG2N>::VALID_OFF);
}
// Batch (S2) mode: the caller supplies the unfiltered border of every PU as the linear 4N+1 array of
// include/cucudecide.h ([0..2N-1] left column bottom -> top, [2N] corner, [2N+1..4N] above row); substitution has
// already happened in the encoder (TComPattern.cpp:314-521).  T[k] = b[2N + k], L[k] = b[2N - k].
template <int LOG2N>
CUCD_HD void build_unfiltered_batch(int tid, int ctu, const int16_t* b /*border of PU tid / TPP, or null*/, unsigned char* smem) {
  typedef Cfg<LOG2N> C;
  constexpr int N = C::N, TPP = 256 / C::PUS, SPT = 4 * N / TPP;
  unsigned char* store = smem + C::STORE_OFF;
  const int p = tid / TPP, sub = tid % TPP;
  if (!smem[C::VALID_OFF + ctu * 256 + p]) return;
  if (LOG2N == 2) {
    auto w4 = [](int b0, int b1, int b2, int b3) { return (uint32_t)(b0 & 255) | ((uint32_t)(b1 & 255) << 8) | ((uint32_t)(b2 & 255) << 16) | ((uint32_t)(b3 & 255) << 24); };
    const int16_t* t = b + 8;                       // t[k] = T[k], t[-k] = L[k]
    uint32_t* r0 = reinterpret_cast<uint32_t*>(store + rec_off(ctu, 0, p));
    uint32_t* r1 = reinterpret_cast<uint32_t*>(store + rec_off(ctu, 1, p));
    r0[0] = w4(t[0], t[1], t[2], t[3]); r0[1] = w4(t[4], t[5], t[6], t[7]); r0[2] = w4(t[8], t[-1], t[-2], t[-3]); r0[3] = w4(t[-4], t[-5], 0, 1);
    r1[0] = w4(t[0], t[-1], t[-2], t[-3]); r1[1] = w4(t[-4], t[-5], t[-6], t[-7]); r1[2] = w4(t[-8], t[1], t[2], t[3]); r1[3] = w4(t[4], t[5], 0, 1);
    return;
  }
  if (sub == 0) { put_ref<LOG2N>(store, ctu, p, 0, 0, b[2 * N]); put_ref<LOG2N>(store, ctu, p, 1, 0, b[2 * N]); }
  int dcSum = 0;
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    const int v = o ? b[2 * N - k] : b[2 * N + k];
    put_ref<LOG2N>(store, ctu, p, o, k, v);
    if (k <= N) dcSum += v;
  }
  int* dst = reinterpret_cast<int*>(smem + C::DC_OFF) + ctu * 64 + p;
#if defined(__CUDA_ARCH__)
  if (dcSum) atomicAdd(dst, dcSum);
#else
  *dst += dcSum;
#endif
}

// Phase 3: smoothed arrays (TComPattern.cpp:185-283) from the unfiltered ones, same thread -> sample map
template <int LOG2N>
CUCD_HD void build_filtered_at(int tid, int ctu, int strongEnabled, unsigned char* prol) {
  typedef Cfg<LOG2N> C;
  if (!C::HAS_FILT) return;
  constexpr int N = C::N, TPP = 256 / C::PUS, SPT = 4 * N / TPP;
  unsigned char* store = prol + ProlOff<LOG2N>::STORE;
  const int p = tid / TPP, sub = tid % TPP;
  if (!prol[ctu * 256 + p]) return;
  const int slot = pu_slot2<LOG2N>(ctu, p);
  const int g0 = LOG2N == 3 ? ctu : 0;
  const unsigned char* T = store + arr_k0_off<LOG2N>(g0, slot, 0, 0);
  const unsigned char* L = store + arr_k0_off<LOG2N>(g0, slot, 1, 0);
  bool strong = false;
  const int tl = T[0], bl = L[2 * N], tr = T[2 * N];
  if (LOG2N == 5 && strongEnabled) strong = iabs32(bl + tl - 2 * (int)L[N]) < 8 && iabs32(tl + tr - 2 * (int)T[N]) < 8;   // 1 << (bitDepth - 5)
  auto put = [&](int o, int k, int v) {
    if (LOG2N == 3) store[arr_k0_off<LOG2N>(ctu, slot, o, 1) + k] = (unsigned char)v;
    else { store[arr_k0_off<LOG2N>(0, slot, o, 1) + k] = (unsigned char)v; store[arr_k0_off<LOG2N>(1, slot, o, 1) + k] = (unsigned char)v; }
  };
  if (sub == 0) {
    const int c = strong ? tl : ((int)L[1] + 2 * tl + (int)T[1] + 2) >> 2;
    put(0, 0, c); put(1, 0, c);
  }
  int vals[SPT];
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    const unsigned char* A = o ? L : T;
    if (k == 2 * N) vals[e] = A[k];
    else if (strong) vals[e] = o ? (k * bl + (2 * N - k) * tl + N) >> (LOG2N + 1) : ((2 * N - k) * tl + k * tr + N) >> (LOG2N + 1);
    else vals[e] = ((int)A[k - 1] + 2 * (int)A[k] + (int)A[k + 1] + 2) >> 2;
  }
#pragma unroll
  for (int e = 0; e < SPT; e++) {
    const int j = sub * SPT + e;
    const int o = j >= 2 * N, k = j - o * 2 * N + 1;
    put(o, k, vals[e]);
  }
}

template <int LOG2N>
CUCD_HD void build_filtered(int tid, int ctu, int strongEnabled, unsigned char* smem) { build_filtered_at<LOG2N>(tid, ctu, strongEnabled, smem + Cfg<LOG2N>::VALID_OFF); }

// projected samples of a negative-angle round, by the 128 threads of row group `grp` for its private arrays:
// store[main][-j] = store[side][(128 + j*inv) >> 8] (TComPrediction.cpp:300-322).  128 / (2 * SLOTS) threads share one
// (slot, orientation) pair; a thread produces N / TPP consecutive entries, four at a time as one aligned 32-bit store.
// ALL N entries of the array are written: those beyond the mode's own -((N * angle) >> 5) - 1 are never consumed by a
// window; their side indices are clamped into the side array.
template <int LOG2N>
CUCD_HD void build_ext_group(int rowTid, int grp, int inv, int filt, unsigned char* store) {
  typedef Cfg<LOG2N> C;
  constexpr int TPP = LOG2N == 2 ? 1 : 128 / (2 * C::SLOTS);   // (N = 4 has no projected arrays; never called)
  constexpr int EPT = C::N / TPP;                              // 8 entries per thread (N = 64: 4)
  static_assert(LOG2N == 2 || EPT % 4 == 0, "entries are produced four at a time");
  const int pair = rowTid / TPP, sub = rowTid % TPP, slot = pair >> 1, o = pair & 1;
  const int mainOff = arr_k0_off<LOG2N>(grp, slot, o, filt);
  const unsigned char* side = store + arr_k0_off<LOG2N>(grp, slot, o ^ 1, filt);
  int t = 128 + (sub * EPT + 1) * inv;                         // 128 + j * inv of the thread's first entry j
  uint32_t* dst = reinterpret_cast<uint32_t*>(store + mainOff - sub * EPT - 4);   // entries j .. j+3 live at bytes 3 .. 0 of this word
#pragma unroll
  for (int q = 0; q < EPT / 4; q++) {
    constexpr int kMax = 2 * C::N;
    const uint32_t b3 = side[imin32(t >> 8, kMax)], b2 = side[imin32((t + inv) >> 8, kMax)], b1 = side[imin32((t + 2 * inv) >> 8, kMax)],
                   b0 = side[imin32((t + 3 * inv) >> 8, kMax)];
    dst[-q] = bperm(bperm(b0, b1, 0x3340), bperm(b2, b3, 0x3340), 0x5410);
    t += 4 * inv;
  }
}

}  // namespace tc2
}  // namespace cucd
