// me_core.cuh - tile decomposition and per-lane arithmetic of the integer-ME SAD surface kernels (me_kernels.cu).
// Host/device so that tests/emul can replay it.  Reference: TComRdCost::xGetSAD* (TComRdCost.cpp:465-962): rows stepped by
// 1 << subShift, sum << subShift, then >> (bitDepth - 8); the candidates are those of TEncSearch::xTZSearchHelp
// (TEncSearch.cpp:336-437) / xPatternSearch (:3886-3943).
//
// A surface (cols x rows candidates of one PU) is cut into three kinds of tiles:
//   M  32 dx x 64 dy, "dy lanes": a lane owns one dy, a warp one byte / half-word alignment of dx, a thread EIGHT candidates
//      dx = x0 + s + stride * k that slide over the same staged reference words: one shared-memory load (+ one PRMT / SHF when the
//      alignment is not 0) feeds eight absolute-difference instructions, the source word is a broadcast load.
//   E  the last 1..4 columns of a window whose width is 32 * n + 1..4 (HM's +-R windows are 2R + 1 wide): dy lanes, one candidate
//      per thread, up to 128 dy per CTA.
//   O  everything else (windows below 32 x 32, the last rows % 32 rows, a right strip wider than 4): the dx-lane tiles of
//      me_sad_kernel / me_sad_u8_kernel.
#pragma once
#include "rmd_core.cuh"

namespace cucd {

constexpr int kMeKindO = 0, kMeKindM = 1, kMeKindE = 2;
constexpr int kMeMaxWindow = 8191;                  // cols, rows of a window (13 bits each in a tile record)
constexpr int kMeDyPitch8 = 25;                     // staged reference row in 32-bit words, 8-bit samples: >= (64 + 31) / 4 + 2, odd (lanes = rows)
constexpr int kMeDyPitch16 = 49;                    // 16-bit samples: >= (64 + 31) / 2 + 2, odd
constexpr int kMeDyRows = 64 + 127;                 // an E tile covers up to 128 dy
constexpr int kMeDyK = 8;                           // candidates per thread in an M tile

CUCD_HD int32_t me_tile_pack(int kind, int x0, int y0) { return (int32_t)((kind << 26) | (y0 << 13) | x0); }
CUCD_HD void me_tile_unpack(int32_t t, int& kind, int& x0, int& y0) { kind = (t >> 26) & 3; y0 = (t >> 13) & 0x1fff; x0 = t & 0x1fff; }
CUCD_HD int me_edge_blocks(int cr) { return 8 / cr < 4 ? 8 / cr : 4; }     // 32-dy blocks of an E tile with cr columns (8 warps)

// the dy-lane kernel unrolls a row by its width: HM's PU widths (TComRdCost.cpp:322-372 has a SAD function for each of them)
CUCD_HD bool me_width_is_hm(int w) { return w == 4 || w == 8 || w == 12 || w == 16 || w == 24 || w == 32 || w == 48 || w == 64; }
// emit(kind, x0, y0) for every tile of a cols x rows window; `fast`: the dy-lane kernel may be used (picture-resident source, unsigned
// samples, one of HM's PU widths)
template <class F>
inline void me_enum_tiles(int cols, int rows, bool fast, int tileRowsO, F&& emit) {
  if (!fast || cols < 32 || rows < 32) {
    for (int y0 = 0; y0 < rows; y0 += tileRowsO) for (int x0 = 0; x0 < cols; x0 += 32) emit(kMeKindO, x0, y0);
    return;
  }
  const int colsMain = cols & ~31, rowsA = rows & ~31, cr = cols - colsMain;
  for (int y0 = 0; y0 < rowsA; y0 += 64) for (int x0 = 0; x0 < colsMain; x0 += 32) emit(kMeKindM, x0, y0);
  if (cr > 0) {
    if (cr <= 4) { const int span = 32 * me_edge_blocks(cr); for (int y0 = 0; y0 < rows; y0 += span) emit(kMeKindE, colsMain, y0); }
    else for (int y0 = 0; y0 < rows; y0 += tileRowsO) emit(kMeKindO, colsMain, y0);
  }
  for (int y0 = rowsA; y0 < rows; y0 += tileRowsO) for (int x0 = 0; x0 < colsMain; x0 += 32) emit(kMeKindO, x0, y0);
}

// geometry of a dy-lane tile (kinds M and E), identical for both sample widths
struct MeDyTile {
  int nLam;        // candidate rows (dy) of the tile
  int winW, winH;  // staged reference window in samples / rows
  int cr;          // E: columns of the strip
};
CUCD_HD MeDyTile me_dy_tile(int kind, int x0, int y0, int w, int h, int cols, int rows) {
  MeDyTile t;
  if (kind == kMeKindM) { const int rowsA = rows & ~31; t.cr = 32; t.nLam = rowsA - y0 < 64 ? rowsA - y0 : 64; t.winW = w + 31; }
  else { t.cr = cols - x0; const int span = 32 * me_edge_blocks(t.cr); t.nLam = rows - y0 < span ? rows - y0 : span; t.winW = w + t.cr - 1; }
  t.winH = h + t.nLam - 1;
  return t;
}
// what a warp of a dy-lane tile does: candidates dx = x0 + delta0 + stride * k (k < K), dy = y0 + 32 * blk + lane
struct MeDyWarp { bool active; int blk, s, wbase, delta0; };
template <bool U8>
CUCD_HD MeDyWarp me_dy_warp(int kind, int warp, int cr) {
  MeDyWarp q;
  if (kind == kMeKindM) {
    q.active = true; q.blk = warp >> 2;
    if (U8) { q.s = warp & 3; q.wbase = 0; q.delta0 = q.s; }                                        // delta = s + 4 k
    else { q.s = warp & 1; q.wbase = 8 * ((warp >> 1) & 1); q.delta0 = q.s + 2 * q.wbase; }         // delta = s + 2 (8 kg + k)
  } else {
    const int col = warp % cr; q.blk = warp / cr; q.active = q.blk < me_edge_blocks(cr); q.delta0 = col;
    if (U8) { q.s = col; q.wbase = 0; } else { q.s = col & 1; q.wbase = col >> 1; }
  }
  return q;
}

// ---- intrinsics with host restatements ---------------------------------------------------------------------------------------
CUCD_HD uint32_t me_prmt_shift(uint32_t lo, uint32_t hi, uint32_t s) {   // bytes s .. s + 3 of the pair {lo, hi}
#if defined(__CUDA_ARCH__)
  return __byte_perm(lo, hi, 0x3210u + 0x1111u * s);
#else
  return s ? (uint32_t)((((uint64_t)hi << 32) | lo) >> (8 * s)) : lo;
#endif
}
CUCD_HD uint32_t me_sad4(uint32_t a, uint32_t b, uint32_t acc) {          // VABSDIFF4.U8.ACC
#if defined(__CUDA_ARCH__)
  uint32_t d;                                                             // __vsadu4(a, b) + acc keeps a separate IADD: the header's asm has a literal 0 addend
  asm("vabsdiff4.u32.u32.u32.add %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(acc));
  return d;
#else
  for (int i = 0; i < 4; i++) { const int x = (a >> (8 * i)) & 255, y = (b >> (8 * i)) & 255; acc += (uint32_t)(x > y ? x - y : y - x); }
  return acc;
#endif
}
CUCD_HD uint32_t me_min2(uint32_t a, uint32_t b) {                        // VIMNMX.S16x2
#if defined(__CUDA_ARCH__)
  return __vmins2(a, b);
#else
  const int16_t al = (int16_t)(a & 0xffffu), ah = (int16_t)(a >> 16), bl = (int16_t)(b & 0xffffu), bh = (int16_t)(b >> 16);
  return (uint32_t)(uint16_t)(al < bl ? al : bl) | ((uint32_t)(uint16_t)(ah < bh ? ah : bh) << 16);
#endif
}
CUCD_HD uint32_t me_fold2(uint32_t packed, uint32_t acc) {                // acc + low half + high half (unsigned IDP.2A)
#if defined(__CUDA_ARCH__)
  return __dp2a_lo(packed, 0x0101u, acc);
#else
  return acc + (packed & 0xffffu) + (packed >> 16);
#endif
}

// ---- per-lane work of a dy-lane tile -------------------------------------------------------------------------------------------
// cw: the PU as words, row y at cw[y * words]; rw: the staged window, row r at rw[r * P]; lam: the lane's candidate row inside the tile.
// Aligned word m of a window row = staged bytes 4 (wbase + m) + s ...; candidate k compares source word j with aligned word j + k.
// The row width is a template parameter (HM's PU widths are 4, 8, 12, 16, 24, 32, 48, 64): a run of N source words is fully
// unrolled - N + K - 1 aligned words in registers, no loop or bounds predicates between the absolute-difference instructions.
template <int K, int N>
CUCD_HD void me_dy_run_u8(const uint32_t* cc, const uint32_t* rr, uint32_t s, uint32_t* acc /*K*/) {
  uint32_t A[N + K - 1];
  uint32_t prev = rr[0];
#pragma unroll
  for (int m = 0; m < N + K - 1; m++) { const uint32_t nx = rr[m + 1]; A[m] = me_prmt_shift(prev, nx, s); prev = nx; }
#pragma unroll
  for (int t = 0; t < N; t++) {
    const uint32_t c = cc[t];
#pragma unroll
    for (int k = 0; k < K; k++) acc[k] = me_sad4(c, A[t + k], acc[k]);
  }
}
template <int K, int WORDS>
CUCD_HD void me_dy_rows_u8(const uint32_t* cw, const uint32_t* rw, int h, int step, int lam, int wbase, int s, uint32_t* acc /*K*/) {
#pragma unroll 1
  for (int y = 0; y < h; y += step) me_dy_run_u8<K, WORDS>(cw + y * WORDS, rw + (lam + y) * kMeDyPitch8 + wbase, (uint32_t)s, acc);
}
template <int K>
CUCD_HD void me_dy_sad_u8(const uint32_t* cw, const uint32_t* rw, int words, int h, int step, int lam, int wbase, int s, uint32_t* acc /*K*/) {
#pragma unroll
  for (int k = 0; k < K; k++) acc[k] = 0;
  switch (words) {
    case 1: me_dy_rows_u8<K, 1>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 2: me_dy_rows_u8<K, 2>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 3: me_dy_rows_u8<K, 3>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 4: me_dy_rows_u8<K, 4>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 6: me_dy_rows_u8<K, 6>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 8: me_dy_rows_u8<K, 8>(cw, rw, h, step, lam, wbase, s, acc); break;
    case 12: me_dy_rows_u8<K, 12>(cw, rw, h, step, lam, wbase, s, acc); break;
    default: me_dy_rows_u8<K, 16>(cw, rw, h, step, lam, wbase, s, acc); break;
  }
}

// 9/10-bit samples as packed int16 pairs, all in [0, 2^bitDepth): sum |c - r| = sum c + sum r - 2 sum min(c, r).  The three sums are
// accumulated per 16-bit half in packed words (one IADD per word, two fused into an IADD3) and folded into 32-bit totals every
// foldRows rows, before a half can exceed 65535: foldRows * pairs * (2^bitDepth - 1) < 65536.
CUCD_HD int me_fold_rows(int bitDepth, int pairs) { const int f = (1 << (16 - bitDepth)) / pairs; return f < 1 ? 1 : f; }
template <int K, int N>                              // a run of N source words (N even: two words per step, the additions pair up into IADD3)
CUCD_HD void me_dy_run_s16(const uint32_t* cc, const uint32_t* rr, uint32_t sh, uint32_t& pA, uint32_t* pM /*K*/, uint32_t* pR /*K*/) {
  uint32_t A[N + K - 1];
  uint32_t prev = rr[0];
#pragma unroll
  for (int m = 0; m < N + K - 1; m++) { const uint32_t nx = rr[m + 1]; A[m] = funnel_r(prev, nx, sh); prev = nx; }
#pragma unroll
  for (int t = 0; t < N; t += 2) {
    const uint32_t c0 = cc[t], c1 = cc[t + 1];
    pA = pA + c0 + c1;
#pragma unroll
    for (int k = 0; k < K; k++) { pM[k] = pM[k] + me_min2(c0, A[t + k]) + me_min2(c1, A[t + 1 + k]); pR[k] = pR[k] + A[t + k] + A[t + 1 + k]; }
  }
}
template <int K, int PAIRS>
CUCD_HD void me_dy_rows_s16(const uint32_t* cw, const uint32_t* rw, int h, int step, int lam, int wbase, int s, int foldRows, uint32_t* sad /*K*/) {
  uint32_t totM[K], totR[K], pM[K], pR[K], totA = 0, pA = 0;
#pragma unroll
  for (int k = 0; k < K; k++) { totM[k] = 0; totR[k] = 0; pM[k] = 0; pR[k] = 0; }
  int pend = 0;
  const uint32_t sh = 16u * (uint32_t)s;
#pragma unroll 1
  for (int y = 0; y < h; y += step) {
    const uint32_t* rr = rw + (lam + y) * kMeDyPitch16 + wbase;
    const uint32_t* cc = cw + y * PAIRS;
    constexpr int R0 = PAIRS > 16 ? 16 : PAIRS;      // runs of at most 16 words keep the aligned words in registers
    me_dy_run_s16<K, R0>(cc, rr, sh, pA, pM, pR);
    if constexpr (PAIRS > 16) me_dy_run_s16<K, PAIRS - R0>(cc + R0, rr + R0, sh, pA, pM, pR);
    if (++pend == foldRows) {
      pend = 0;
      totA = me_fold2(pA, totA); pA = 0;
#pragma unroll
      for (int k = 0; k < K; k++) { totM[k] = me_fold2(pM[k], totM[k]); totR[k] = me_fold2(pR[k], totR[k]); pM[k] = 0; pR[k] = 0; }
    }
  }
  totA = me_fold2(pA, totA);
#pragma unroll
  for (int k = 0; k < K; k++) sad[k] = totA + me_fold2(pR[k], totR[k]) - 2u * me_fold2(pM[k], totM[k]);
}
template <int K>
CUCD_HD void me_dy_sad_s16(const uint32_t* cw, const uint32_t* rw, int pairs, int h, int step, int lam, int wbase, int s, int foldRows, uint32_t* sad /*K*/) {
  switch (pairs) {
    case 2: me_dy_rows_s16<K, 2>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 4: me_dy_rows_s16<K, 4>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 6: me_dy_rows_s16<K, 6>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 8: me_dy_rows_s16<K, 8>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 12: me_dy_rows_s16<K, 12>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 16: me_dy_rows_s16<K, 16>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    case 24: me_dy_rows_s16<K, 24>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
    default: me_dy_rows_s16<K, 32>(cw, rw, h, step, lam, wbase, s, foldRows, sad); break;
  }
}

// ---- staging of a dy-lane tile (every thread of the CTA; tid = 32 * warp + lane) ---------------------------------------------------
// source: rows y = 0, step, 2 step, ... of the PU at cur (stride curStride) -> cw[y * (w / spw) + ...], spw samples per word
template <bool U8>
CUCD_HD void me_dy_stage_cur(int warp, int lane, const int16_t* cur, int curStride, int w, int h, int step, uint32_t* cw) {
  constexpr int SPW = U8 ? 4 : 2;
  const int words = w / SPW;
  for (int y = warp * step; y < h; y += 8 * step)
    for (int q = lane; q < words; q += 32) {
      const int16_t* p = cur + (size_t)y * curStride + q * SPW;
      cw[y * words + q] = U8 ? ((uint32_t)(uint8_t)p[0] | ((uint32_t)(uint8_t)p[1] << 8) | ((uint32_t)(uint8_t)p[2] << 16) | ((uint32_t)(uint8_t)p[3] << 24))
                             : ((uint32_t)(uint16_t)p[0] | ((uint32_t)(uint16_t)p[1] << 16));
    }
}
// reference window: winH rows of winW samples starting at ref (stride refStride); the words a candidate's PRMT / SHF touches beyond
// winW are zero filled, nothing outside the window is read
template <bool U8>
CUCD_HD void me_dy_stage_ref(int warp, int lane, const int16_t* ref, long long refStride, int winW, int winH, uint32_t* rw) {
  constexpr int SPW = U8 ? 4 : 2, P = U8 ? kMeDyPitch8 : kMeDyPitch16;
  int wp = (winW + SPW - 1) / SPW + 1;
  if (wp > P) wp = P;
  int lg = 0;
  while ((1 << lg) < wp) lg++;                       // a warp takes 32 >> lg rows at a time (narrow PUs: 2 or 4 rows per pass)
  const int rpw = lg < 5 ? 32 >> lg : 1, lanesPerRow = lg < 5 ? 1 << lg : 32;
  const int rs = lane >> (lg < 5 ? lg : 5), q0 = lane & (lanesPerRow - 1);
  for (int r = warp * rpw + rs; r < winH; r += 8 * rpw)
    for (int q = q0; q < wp; q += lanesPerRow) {
      const int16_t* p = ref + (long long)r * refStride + q * SPW;
      uint32_t v = 0;
#pragma unroll
      for (int i = 0; i < SPW; i++)
        if (q * SPW + i < winW) v |= (U8 ? (uint32_t)(uint8_t)p[i] : (uint32_t)(uint16_t)p[i]) << ((U8 ? 8 : 16) * i);
      rw[r * P + q] = v;
    }
}

// =============================================================================================================================
// Fractional-pel refinement of small PUs (w * h <= 256): ONE CTA per PU evaluates all 49 quarter-pel positions.
// me_subpel_kernel gives a CTA one PU and one horizontal offset; for an 8x8 PU that is 64 samples and 8 Hadamard lanes per pass of a
// 256-thread CTA, and every pass still costs all eight warps their loop and barrier overhead.  Here the seven horizontally filtered
// planes of the PU are built together (7 (h + 9) w intermediates), and the column filter, the distortion and the sums run over
// GROUPS of positions (as many as fit 4096 predicted samples: all 49 for an 8x8 PU, 16 for a 16x16 PU), one thread per sample /
// per Hadamard tile.  Same arithmetic as me_subpel_kernel (TComInterpolationFilter.cpp:57-290, TComRdCost.cpp:1343-1534); the
// Hadamard is satd8x8_packed / satd4x4_packed of rmd_core.cuh on the packed residual (picture-resident sources only: samples in
// [0, 2^bitDepth), so that the packed halves stay inside int16 - caller-supplied key blocks keep me_subpel_kernel).
// =============================================================================================================================
constexpr int kSpSmallWinCap = 1024;      // (h + 9) x (w + 10) int16, max 73 x 14 (4 x 64 PU)
constexpr int kSpHorCap = 73 * 64;        // seven planes of (h + 9) x w intermediates must fit this
constexpr int kSpPredCap = 4096;
CUCD_HD bool subpel_is_small(int w, int h) { return w * h <= 256 && 7 * (h + 9) * w <= kSpHorCap; }
CUCD_HD uint32_t me_inv(uint32_t d) { return 0xffffffffu / d + 1u; }                     // n / d == mulhi(n, me_inv(d)) while n * d < 2^32
CUCD_HD uint32_t me_mulhi(uint32_t n, uint32_t m) {
#if defined(__CUDA_ARCH__)
  return __umulhi(n, m);
#else
  return (uint32_t)(((uint64_t)n * m) >> 32);
#endif
}
CUCD_HD uint32_t me_ld_pair(const int16_t* p) {                                        // two int16 at an even index as one word
#if defined(__CUDA_ARCH__)
  return *reinterpret_cast<const uint32_t*>(p);
#else
  return (uint32_t)(uint16_t)p[0] | ((uint32_t)(uint16_t)p[1] << 16);
#endif
}
// sum s[(k - 3) * stride] * lumaFilter[frac][k], frac = 1..3 (TComInterpolationFilter.cpp:57-63)
CUCD_HD int luma_filter8(const int16_t* s, int stride, int frac) {
  const int a = s[-3 * stride], b = s[-2 * stride], c = s[-stride], d = s[0], e = s[stride], f = s[2 * stride], g = s[3 * stride], h = s[4 * stride];
  if (frac == 1) return -a + 4 * b - 10 * c + 58 * d + 17 * e - 5 * f + g;
  if (frac == 2) return -a + 4 * b - 11 * c + 40 * d + 40 * e - 11 * f + 4 * g - h;
  return b - 5 * c + 17 * d + 58 * e - 10 * f + 4 * g - h;
}
struct SubpelGeo {
  int w, h, bd, head, wh, plane /* (h + 9) * w */, pitch /* w + 10 */;
  uint32_t invW, invWh, invPlane, invPitch;
};
CUCD_HD SubpelGeo subpel_geo(int w, int h, int bd) {
  SubpelGeo g;
  g.w = w; g.h = h; g.bd = bd; g.head = 14 - bd; g.wh = w * h; g.plane = (h + 9) * w; g.pitch = w + 10;
  g.invW = me_inv((uint32_t)w); g.invWh = me_inv((uint32_t)g.wh); g.invPlane = me_inv((uint32_t)g.plane); g.invPitch = me_inv((uint32_t)(w + 9));
  return g;
}
// source block and the (w + 9) x (h + 9) window whose origin is (-4, -4) from the integer MV position
CUCD_HD void subpel_small_stage(int tid, const SubpelGeo& g, const int16_t* cur, int curStride, const int16_t* refWin, long long refStride, int16_t* sCur, int16_t* sWin) {
  for (int i = tid; i < g.wh; i += 256) { const int y = (int)me_mulhi((uint32_t)i, g.invW), x = i - y * g.w; sCur[i] = cur[(size_t)y * curStride + x]; }
  for (int i = tid; i < (g.h + 9) * (g.w + 9); i += 256) {
    const int y = (int)me_mulhi((uint32_t)i, g.invPitch), x = i - y * (g.w + 9);
    sWin[y * g.pitch + x] = refWin[(long long)y * refStride + x];
  }
}
// rows -> 14-bit intermediates for the seven horizontal offsets dx = -3..3 (filterHor, isFirst, !isLast): sHor[dxi][r][c]
CUCD_HD void subpel_small_hor(int tid, const SubpelGeo& g, const int16_t* sWin, int16_t* sHor) {
  for (int i = tid; i < 7 * g.plane; i += 256) {
    const int dxi = (int)me_mulhi((uint32_t)i, g.invPlane), rem = i - dxi * g.plane;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const int dx = dxi - 3, ix = dx >> 2, fx = dx & 3;
    const int16_t* s = &sWin[r * g.pitch + c + 4 + ix];
    const int v = fx == 0 ? (s[0] << g.head) - 8192 : (luma_filter8(s, 1, fx) - (8192 << (6 - g.head))) >> (6 - g.head);
    sHor[i] = (int16_t)v;
  }
}
// columns (filterVer, !isFirst, isLast) for the positions pBase .. pBase + nP - 1 (position p = (dy + 3) * 7 + dx + 3): sPred[pl][r][c]
CUCD_HD void subpel_small_ver(int tid, const SubpelGeo& g, int pBase, int nP, const int16_t* sHor, int16_t* sPred) {
  const uint32_t inv7 = me_inv(7u);
  for (int i = tid; i < nP * g.wh; i += 256) {
    const int pl = (int)me_mulhi((uint32_t)i, g.invWh), rem = i - pl * g.wh;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const int p = pBase + pl, dyi = (int)me_mulhi((uint32_t)p, inv7), dxi = p - 7 * dyi;
    const int dy = dyi - 3, iy = dy >> 2, fy = dy & 3;
    const int16_t* s = &sHor[dxi * g.plane + (r + 4 + iy) * g.w + c];
    int v = fy == 0 ? (s[0] + 8192 + (1 << (g.head - 1))) >> g.head : (luma_filter8(s, g.w, fy) + (1 << (5 + g.head)) + (8192 << 6)) >> (6 + g.head);
    v = v < 0 ? 0 : (v > (1 << g.bd) - 1 ? (1 << g.bd) - 1 : v);
    sPred[i] = (int16_t)v;
  }
}
CUCD_HD void me_smem_add(int* where, int what) {       // shared-memory atomic in the kernel, a plain addition in the CPU replay
#if defined(__CUDA_ARCH__)
  atomicAdd(where, what);
#else
  *where += what;
#endif
}
// distortion of the nP predicted blocks: xGetHADs (8x8 tiles when both sizes are multiples of 8, else 4x4) or xGetSAD, one thread per
// tile / per sample.  curPlane: 0 = one source block for every prediction (the 49 positions of one PU), wh = block pl has its own
// source block at sCur + pl * wh (the candidates of me_mc_kernel)
CUCD_HD void subpel_small_dist(int tid, const SubpelGeo& g, int nP, int useHadamard, const int16_t* sCur, const int16_t* sPred, int* sSum, int curPlane = 0) {
  if (useHadamard) {
    const bool tile8 = !(g.w & 7) && !(g.h & 7);
    const int T = tile8 ? 8 : 4, tilesX = g.w / T, nTiles = tilesX * (g.h / T);
    for (int task = tid; task < nP * nTiles; task += 256) {
      const int pl = task / nTiles, tile = task - pl * nTiles, ty = tile / tilesX, tx = tile - ty * tilesX;
      const int16_t* a = sCur + pl * curPlane + ty * T * g.w + tx * T;
      const int16_t* b = sPred + pl * g.wh + ty * T * g.w + tx * T;
      uint32_t cost;
      if (tile8) {
        uint32_t d[32];
#pragma unroll
        for (int y = 0; y < 8; y++)
#pragma unroll
          for (int j = 0; j < 4; j++) d[y * 4 + j] = me_ld_pair(a + y * g.w + 2 * j) - me_ld_pair(b + y * g.w + 2 * j);
        cost = satd8x8_packed(d);
      } else {
        uint32_t d[8];
#pragma unroll
        for (int y = 0; y < 4; y++)
#pragma unroll
          for (int j = 0; j < 2; j++) d[y * 2 + j] = me_ld_pair(a + y * g.w + 2 * j) - me_ld_pair(b + y * g.w + 2 * j);
        cost = satd4x4_packed(d);
      }
      me_smem_add(&sSum[pl], (int)cost);
    }
  } else {
    for (int i = tid; i < nP * g.wh; i += 256) {
      const int pl = (int)me_mulhi((uint32_t)i, g.invWh);
      const int d = iabs32((int)sCur[i - pl * g.wh + pl * curPlane] - (int)sPred[i]);
      if (d) me_smem_add(&sSum[pl], d);
    }
  }
}

// =============================================================================================================================
// Motion compensation and distortion of inter candidates (cucd_me_mc_cost): TComPrediction::motionCompensation for luma
// (xPredInterUni / xPredInterBi -> xPredInterBlk, TComPrediction.cpp:496-620; TComInterpolationFilter.cpp:57-290 filter /
// filterCopy; TComYuv::addAvg, TComYuv.cpp:260-310) followed by the DistFunc of xGetInterPredictionError (TEncSearch.cpp:2905-2926,
// iSubShift = 0).  A candidate is one PU at one quarter-pel motion of one list (uni) or two lists (bi).  The host sorts the
// candidates into classes of equal shape, list count and distortion; a CTA takes up to me_mc_per_cta() candidates of one class, so
// that every phase maps a flat index onto (candidate, list, row, column) with multiply-high divisions and small PUs share a CTA.
//   stage  the source blocks and, per candidate and list, the (w + 7) x (h + 7) reference window whose origin is (-3, -3) from the
//          integer part of the MV
//   hor    rows -> 14-bit intermediates (filterHor, isFirst, !isLast; filterCopy isFirst for a zero fraction), h + 7 rows per list
//   ver    columns.  Uni: filterVer (!isFirst, isLast) with rounding and clipping, as subpel_small_ver.  Bi: filterVer (!isFirst,
//          !isLast) - sum >> 6, a plain copy at fraction 0 - per list, then addAvg: clip((p0 + p1 + 2^(14-bd) + 16384) >> (15-bd)).
//          The predictions overwrite the dead windows.
//   dist   subpel_small_dist on the candidates' own source blocks
// =============================================================================================================================
constexpr int kMcCurCap = 4096;           // source blocks (and predictions) of a CTA, int16
constexpr int kMcWinCap = 10240;          // reference windows: sum over candidates and lists of (w + 7) (h + 7), >= 2 * 71 * 71
constexpr int kMcTmpCap = 9216;           // row intermediates: sum of (h + 7) w, >= 2 * 71 * 64
constexpr int kMcMaxCand = 64;            // candidates of a CTA
CUCD_HD int me_mc_per_cta(int w, int h, int nl) {
  int k = kMcCurCap / (w * h);
  const int kw = kMcWinCap / (nl * (w + 7) * (h + 7)), kt = kMcTmpCap / (nl * (h + 7) * w);
  k = k < kw ? k : kw; k = k < kt ? k : kt;
  return k < kMcMaxCand ? k : kMcMaxCand;
}
// CTAs hold candidates of one class: shape, list count and distortion function
inline int me_mc_class(int w, int h, int nl, int had) { return (((((w >> 2) - 1) * 16 + (h >> 2) - 1) * 2 + nl - 1) * 2) + (had ? 1 : 0); }
constexpr int kMcClasses = 16 * 16 * 4;

struct McJob {
  int32_t curOff;      // PU origin inside the current picture plane
  int32_t refOff[2];   // per list: the window origin (-3, -3 from the integer MV position) inside the padded plane of refSlot
  int16_t refSlot[2];
  int8_t fx[2], fy[2]; // per list: quarter-pel fractions
  int16_t w, h;
  int8_t nl, had;      // lists used (1 uni, 2 bi; list 1 of a uni L1 candidate sits in entry 0); xGetHADs / xGetSAD
  int16_t pad;
  int32_t outIndex;    // candidate index in the caller's order (dist)
  int64_t predOff;     // offset of its w x h prediction block in the caller's pred array
};
// host: the job of a candidate whose nl used lists (compacted: entry 0, then entry 1) have reference slot, quarter-pel MV and padded
// plane stride / margins slot[l], mvx[l], mvy[l], stride[l], mX[l], mY[l]
inline McJob me_mc_job(int curOff, int x, int y, int w, int h, int nl, const int* slot, const int* mvx, const int* mvy, const int* stride, const int* mX,
                       const int* mY, int had, int outIndex, long long predOff) {
  McJob j;
  j.curOff = curOff;
  for (int l = 0; l < 2; l++) {
    const int u = l < nl ? l : 0;
    j.refOff[l] = (y + (mvy[u] >> 2) - 3 + mY[u]) * stride[u] + x + (mvx[u] >> 2) - 3 + mX[u];
    j.refSlot[l] = (int16_t)slot[u]; j.fx[l] = (int8_t)(mvx[u] & 3); j.fy[l] = (int8_t)(mvy[u] & 3);
  }
  j.w = (int16_t)w; j.h = (int16_t)h; j.nl = (int8_t)nl; j.had = (int8_t)(had ? 1 : 0); j.pad = 0;
  j.outIndex = outIndex; j.predOff = predOff;
  return j;
}
// host: the jobs sorted by class (cls(job) < NC) into `sorted`, every class cut into CTAs of per(job) jobs; CTA b takes
// sorted[ctaFirst[b] .. ctaFirst[b + 1]).  ctaFirst has room for n + 1 entries; returns the number of CTAs.
template <int NC, class Cls, class Per>
inline int me_plan_classes(int n, const McJob* jobs, McJob* sorted, int32_t* ctaFirst, Cls cls, Per per) {
  int start[NC + 1] = {0};
  for (int i = 0; i < n; i++) start[cls(jobs[i]) + 1]++;
  for (int c = 0; c < NC; c++) start[c + 1] += start[c];
  // stable scatter: start[c] advances to the end of class c
  for (int i = 0; i < n; i++) sorted[start[cls(jobs[i])]++] = jobs[i];
  int nCta = 0;
  for (int b = 0; b < n;) {
    const McJob& j = sorted[b];
    const int e = start[cls(j)], k = per(j);
    for (; b < e; b += k) ctaFirst[nCta++] = b;
    b = e;
  }
  ctaFirst[nCta] = n;
  return nCta;
}
inline int me_mc_plan(int n, const McJob* jobs, McJob* sorted, int32_t* ctaFirst) {
  return me_plan_classes<kMcClasses>(n, jobs, sorted, ctaFirst, [](const McJob& j) { return me_mc_class(j.w, j.h, j.nl, j.had); },
                                     [](const McJob& j) { return me_mc_per_cta(j.w, j.h, j.nl); });
}
struct McGeo {
  int w, h, bd, head, nl, n, wh, pw /* w + 7 (chroma: w + 3) */, win /* pw (h + 7 | h + 3) */, tmp /* (h + 7 | h + 3) w */;
  uint32_t invW, invPw, invWh, invWin, invTmp;
};
CUCD_HD McGeo me_mc_geo(int w, int h, int nl, int n, int bd) {
  McGeo g;
  g.w = w; g.h = h; g.bd = bd; g.head = 14 - bd; g.nl = nl; g.n = n; g.wh = w * h; g.pw = w + 7; g.win = (w + 7) * (h + 7); g.tmp = (h + 7) * w;
  g.invW = me_inv((uint32_t)w); g.invPw = me_inv((uint32_t)g.pw); g.invWh = me_inv((uint32_t)g.wh); g.invWin = me_inv((uint32_t)g.win); g.invTmp = me_inv((uint32_t)g.tmp);
  return g;
}
// every index below is < 10240 and every divisor <= 5041: i * d < 2^32, so the multiply-high divisions are exact
CUCD_HD void me_mc_stage(int tid, const McGeo& g, const McJob* jobs, const int16_t* cur, int curStride, const int16_t* const* ref, const int32_t* refStride,
                         int16_t* sCur, int16_t* sWin) {
  for (int i = tid; i < g.n * g.wh; i += 256) {
    const int k = (int)me_mulhi((uint32_t)i, g.invWh), rem = i - k * g.wh;
    const int y = (int)me_mulhi((uint32_t)rem, g.invW), x = rem - y * g.w;
    sCur[i] = cur[jobs[k].curOff + (long long)y * curStride + x];
  }
  for (int i = tid; i < g.n * g.nl * g.win; i += 256) {
    const int kl = (int)me_mulhi((uint32_t)i, g.invWin), rem = i - kl * g.win;
    const int y = (int)me_mulhi((uint32_t)rem, g.invPw), x = rem - y * g.pw;
    const McJob& j = jobs[kl >> (g.nl - 1)];
    const int l = kl & (g.nl - 1), slot = j.refSlot[l];
    sWin[i] = ref[slot][j.refOff[l] + (long long)y * refStride[slot] + x];
  }
}
// rows of every window -> sTmp[kl][r][c], r = 0 .. h + 6 (filterHor, isFirst, !isLast; filterCopy isFirst at fx = 0)
CUCD_HD void me_mc_hor(int tid, const McGeo& g, const McJob* jobs, const int16_t* sWin, int16_t* sTmp) {
  for (int i = tid; i < g.n * g.nl * g.tmp; i += 256) {
    const int kl = (int)me_mulhi((uint32_t)i, g.invTmp), rem = i - kl * g.tmp;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const int fx = jobs[kl >> (g.nl - 1)].fx[kl & (g.nl - 1)];
    const int16_t* s = &sWin[kl * g.win + r * g.pw + c + 3];
    sTmp[i] = (int16_t)(fx == 0 ? (s[0] << g.head) - 8192 : (luma_filter8(s, 1, fx) - (8192 << (6 - g.head))) >> (6 - g.head));
  }
}
// columns -> the clipped prediction sPred[k][r][c] (and pred[predOff + r w + c] when pred is not null).
// Bi: HM reaches the 14-bit intermediate of a list through four branches of xPredInterBlk (TComPrediction.cpp:560-600): filterCopy
// (isFirst, !isLast) for fx = fy = 0, filterHor (isFirst, !isLast) for fy = 0, filterVer (isFirst, !isLast) on the reference for
// fx = 0, and filterHor (isFirst, !isLast) + filterVer (!isFirst, !isLast) otherwise.  The two-stage form below equals all four:
// the first three are it with a plain-copy second stage or (fx = 0, fy != 0) with taps summing to 64 over s << head - 8192, where
// (sum c (s << head) - 8192 * 64) >> 6 == (sum c s - (8192 << (6 - head))) >> (6 - head) because 2^head divides both numerator
// and divisor.  Intermediates stay in int16: |stage 1| <= 14 330, |stage 2| <= 25 072 at 10 bits; the sums are int32.
CUCD_HD void me_mc_ver(int tid, const McGeo& g, const McJob* jobs, const int16_t* sTmp, int16_t* sPred, int16_t* pred) {
  const int maxVal = (1 << g.bd) - 1;
  for (int i = tid; i < g.n * g.wh; i += 256) {
    const int k = (int)me_mulhi((uint32_t)i, g.invWh), rem = i - k * g.wh;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const McJob& j = jobs[k];
    int v;
    if (g.nl == 1) {
      const int16_t* s = &sTmp[k * g.tmp + (r + 3) * g.w + c];
      const int fy = j.fy[0];
      v = fy == 0 ? (s[0] + 8192 + (1 << (g.head - 1))) >> g.head : (luma_filter8(s, g.w, fy) + (1 << (5 + g.head)) + (8192 << 6)) >> (6 + g.head);
    } else {
      int p[2];
#pragma unroll
      for (int l = 0; l < 2; l++) {
        const int16_t* s = &sTmp[(2 * k + l) * g.tmp + (r + 3) * g.w + c];
        const int fy = j.fy[l];
        p[l] = fy == 0 ? s[0] : luma_filter8(s, g.w, fy) >> 6;
      }
      v = (p[0] + p[1] + (1 << g.head) + 16384) >> (g.head + 1);
    }
    v = v < 0 ? 0 : (v > maxVal ? maxVal : v);
    sPred[i] = (int16_t)v;
    if (pred) pred[j.predOff + rem] = (int16_t)v;
  }
}

// =============================================================================================================================
// 4:2:0 chroma motion compensation and SSE of inter candidates (cucd_me_mc_chroma): the chroma branch of xPredInterBlk
// (TComInterpolationFilter::m_chromaFilter, filterHor / filterVer with 4 taps at p - 1 .. p + 2), TComYuv::addAvg for bi, and the
// getDistPart SSE of encodeResAndCalcRdInterCU, before the chroma weight.  Same layout as the luma kernel: McJob records (w, h, x, y
// in chroma samples, eighth-pel fractions 0..7, had = 0) sorted into classes of equal chroma shape and list count, a CTA takes
// me_mcc_per_cta() candidates of one class, and both planes of a candidate go to the same CTA as plane-candidates p = 2 k + plane.
//   stage  the Cb / Cr source blocks and, per plane-candidate and list, the (w + 3) x (h + 3) window at (-1, -1) from the integer MV
//   hor    rows -> 14-bit intermediates, h + 3 rows per list
//   ver    columns, uni: rounded and clipped; bi: sum >> 6 per list, then addAvg.  The predictions overwrite the dead windows.
//   sse    sum ((org - pred)^2 >> 2 (bd - 8)) per plane-candidate
// Both passes run the 4-tap filter at every fraction: m_chromaFilter[0] = {0, 64, 0, 0} turns it into the copy.  The two-stage form
// equals the four xPredInterBlk branches by the argument beside me_mc_ver, which only needs taps that sum to 64: stage 1 is
// (sum c s - (8192 << (6 - head))) >> (6 - head) ((s << head) - 8192 at fraction 0, filterCopy isFirst); stage 2 is filterVer
// (!isFirst) on it, and for fy = 0 (and fx = 0) the sum over taps {0, 64, 0, 0} leaves the single-stage results of filterHor
// (isFirst, isLast) and filterVer (isFirst, !bi) unchanged, because 2^head divides every term that is dropped.
// Intermediate bounds (exact over the eight filters, head = 14 - bd): stage 1 in [-10 750, 10 733] and the bi stage 2 in
// [-14 107, 14 089] at 10 bits, less at 8 and 9 bits: both int16; the sums are int32.  SSE of a 32 x 32 plane < 2^27: an int counter.
// =============================================================================================================================
// every class: chroma w, h in 2, 4, .., 32 and 1 or 2 lists
constexpr int kMccClasses = 16 * 16 * 2;
inline int me_mcc_class(int w, int h, int nl) { return (((w >> 1) - 1) * 16 + (h >> 1) - 1) * 2 + nl - 1; }
// the caps of the luma kernel, two plane-candidates per candidate
CUCD_HD int me_mcc_per_cta(int w, int h, int nl) {
  int k = kMcCurCap / (2 * w * h);
  const int kw = kMcWinCap / (2 * nl * (w + 3) * (h + 3)), kt = kMcTmpCap / (2 * nl * (h + 3) * w);
  k = k < kw ? k : kw; k = k < kt ? k : kt;
  return k < kMcMaxCand ? k : kMcMaxCand;
}
// host: the job of a candidate's chroma block (x, y, w, h: the luma PU >> 1), luma quarter-pel = chroma eighth-pel MVs; slot, mvx, mvy,
// stride, mX, mY per used list as for me_mc_job, the strides and margins those of the slot's chroma planes
inline McJob me_mcc_job(int curOff, int x, int y, int w, int h, int nl, const int* slot, const int* mvx, const int* mvy, const int* stride, const int* mX,
                        const int* mY, int outIndex, long long predOff) {
  McJob j;
  j.curOff = curOff;
  for (int l = 0; l < 2; l++) {
    const int u = l < nl ? l : 0;
    j.refOff[l] = (y + (mvy[u] >> 3) - 1 + mY[u]) * stride[u] + x + (mvx[u] >> 3) - 1 + mX[u];
    j.refSlot[l] = (int16_t)slot[u]; j.fx[l] = (int8_t)(mvx[u] & 7); j.fy[l] = (int8_t)(mvy[u] & 7);
  }
  j.w = (int16_t)w; j.h = (int16_t)h; j.nl = (int8_t)nl; j.had = 0; j.pad = 0;
  j.outIndex = outIndex; j.predOff = predOff;
  return j;
}
inline int me_mcc_plan(int n, const McJob* jobs, McJob* sorted, int32_t* ctaFirst) {
  return me_plan_classes<kMccClasses>(n, jobs, sorted, ctaFirst, [](const McJob& j) { return me_mcc_class(j.w, j.h, j.nl); },
                                      [](const McJob& j) { return me_mcc_per_cta(j.w, j.h, j.nl); });
}
CUCD_HD McGeo me_mcc_geo(int w, int h, int nl, int n, int bd) {
  McGeo g;
  g.w = w; g.h = h; g.bd = bd; g.head = 14 - bd; g.nl = nl; g.n = n; g.wh = w * h; g.pw = w + 3; g.win = (w + 3) * (h + 3); g.tmp = (h + 3) * w;
  g.invW = me_inv((uint32_t)w); g.invPw = me_inv((uint32_t)g.pw); g.invWh = me_inv((uint32_t)g.wh); g.invWin = me_inv((uint32_t)g.win); g.invTmp = me_inv((uint32_t)g.tmp);
  return g;
}
// sum s[(k - 1) * stride] * m_chromaFilter[frac][k], frac = 0..7:
//   {0, 64, 0, 0} {-2, 58, 10, -2} {-4, 54, 16, -2} {-6, 46, 28, -4} {-4, 36, 36, -4} {-4, 28, 46, -6} {-2, 16, 54, -4} {-2, 10, 58, -2}
// held as byte lanes of three constants (|c0|, c1, |c3|; c2 = 64 - c1 + |c0| + |c3|), so a warp whose lanes see different fractions
// does not branch
CUCD_HD int chroma_filter4(const int16_t* s, int stride, int frac) {
  const int sh = 8 * frac;
  const int n0 = (int)((0x0202040406040200ull >> sh) & 0xff), c1 = (int)((0x0a101c242e363a40ull >> sh) & 0xff), n3 = (int)((0x0204060404020200ull >> sh) & 0xff);
  return -n0 * s[-stride] + c1 * s[0] + (64 - c1 + n0 + n3) * s[stride] - n3 * s[2 * stride];
}
// every index below is < 10240 and every divisor <= 35 * 35: the multiply-high divisions are exact.  cur[plane]: the current
// picture's Cb / Cr plane; ref[2 slot + plane]: the first sample of slot's padded Cb / Cr plane, refStride[slot] of both
CUCD_HD void me_mcc_stage(int tid, const McGeo& g, const McJob* jobs, const int16_t* const* cur, int curStride, const int16_t* const* ref, const int32_t* refStride,
                          int16_t* sCur, int16_t* sWin) {
  for (int i = tid; i < 2 * g.n * g.wh; i += 256) {
    const int p = (int)me_mulhi((uint32_t)i, g.invWh), rem = i - p * g.wh;
    const int y = (int)me_mulhi((uint32_t)rem, g.invW), x = rem - y * g.w;
    const int16_t* c = (p & 1) ? cur[1] : cur[0];                                      // a select, not an indexed (local-memory) copy of the array
    sCur[i] = c[jobs[p >> 1].curOff + (long long)y * curStride + x];
  }
  for (int i = tid; i < 2 * g.n * g.nl * g.win; i += 256) {
    const int pl = (int)me_mulhi((uint32_t)i, g.invWin), rem = i - pl * g.win;          // pl = (2 k + plane) nl + l
    const int y = (int)me_mulhi((uint32_t)rem, g.invPw), x = rem - y * g.pw;
    const int p = pl >> (g.nl - 1), l = pl & (g.nl - 1);
    const McJob& j = jobs[p >> 1];
    const int slot = j.refSlot[l];
    sWin[i] = ref[2 * slot + (p & 1)][j.refOff[l] + (long long)y * refStride[slot] + x];
  }
}
// rows of every window -> sTmp[pl][r][c], r = 0 .. h + 2 (filterHor, isFirst, !isLast)
CUCD_HD void me_mcc_hor(int tid, const McGeo& g, const McJob* jobs, const int16_t* sWin, int16_t* sTmp) {
  for (int i = tid; i < 2 * g.n * g.nl * g.tmp; i += 256) {
    const int pl = (int)me_mulhi((uint32_t)i, g.invTmp), rem = i - pl * g.tmp;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const int fx = jobs[pl >> g.nl].fx[pl & (g.nl - 1)];
    sTmp[i] = (int16_t)((chroma_filter4(&sWin[pl * g.win + r * g.pw + c + 1], 1, fx) - (8192 << (6 - g.head))) >> (6 - g.head));
  }
}
// columns -> the clipped prediction sPred[p][r][c]; pred (may be null) holds a candidate's Cb block, then its Cr block, at predOff
CUCD_HD void me_mcc_ver(int tid, const McGeo& g, const McJob* jobs, const int16_t* sTmp, int16_t* sPred, int16_t* pred) {
  const int maxVal = (1 << g.bd) - 1;
  for (int i = tid; i < 2 * g.n * g.wh; i += 256) {
    const int p = (int)me_mulhi((uint32_t)i, g.invWh), rem = i - p * g.wh;
    const int r = (int)me_mulhi((uint32_t)rem, g.invW), c = rem - r * g.w;
    const McJob& j = jobs[p >> 1];
    int v;
    if (g.nl == 1) {
      v = (chroma_filter4(&sTmp[p * g.tmp + (r + 1) * g.w + c], g.w, j.fy[0]) + (1 << (5 + g.head)) + (8192 << 6)) >> (6 + g.head);
    } else {
      const int p0 = chroma_filter4(&sTmp[2 * p * g.tmp + (r + 1) * g.w + c], g.w, j.fy[0]) >> 6;
      const int p1 = chroma_filter4(&sTmp[(2 * p + 1) * g.tmp + (r + 1) * g.w + c], g.w, j.fy[1]) >> 6;
      v = (p0 + p1 + (1 << g.head) + 16384) >> (g.head + 1);
    }
    v = v < 0 ? 0 : (v > maxVal ? maxVal : v);
    sPred[i] = (int16_t)v;
    if (pred) pred[j.predOff + (long long)(p & 1) * g.wh + rem] = (int16_t)v;
  }
}
// getDistPart (TComRdCost::xGetSSE): sSum[p] += (org - pred)^2 >> 2 (bd - 8)
CUCD_HD void me_mcc_sse(int tid, const McGeo& g, const int16_t* sCur, const int16_t* sPred, int* sSum) {
  const int shift = 2 * (g.bd - 8);
  for (int i = tid; i < 2 * g.n * g.wh; i += 256) {
    const int d = (int)sCur[i] - (int)sPred[i], v = (d * d) >> shift;
    if (v) me_smem_add(&sSum[me_mulhi((uint32_t)i, g.invWh)], v);
  }
}

}  // namespace cucd
