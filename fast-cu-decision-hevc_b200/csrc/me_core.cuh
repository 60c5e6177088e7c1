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
template <int NC, class Job, class Cls, class Per>
inline int me_plan_classes(int n, const Job* jobs, Job* sorted, int32_t* ctaFirst, Cls cls, Per per) {
  int start[NC + 1] = {0};
  for (int i = 0; i < n; i++) start[cls(jobs[i]) + 1]++;
  for (int c = 0; c < NC; c++) start[c + 1] += start[c];
  // stable scatter: start[c] advances to the end of class c
  for (int i = 0; i < n; i++) sorted[start[cls(jobs[i])]++] = jobs[i];
  int nCta = 0;
  for (int b = 0; b < n;) {
    const Job& j = sorted[b];
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

// =============================================================================================================================
// Motion search (cucd_me_search): HM's full search xPatternSearch (TEncSearch.cpp:3886-3943) and the refinement walk of
// xPatternSearchFracDIF / xPatternRefinement (:4340-4376, :808-865) on top of the SAD surface and sub-pel table arithmetic.
//   integer  the SAD kernels in their Argmin form: a candidate becomes the key ((sad + cost_2(mv)) << 32) | (dy * cols + dx), a
//            warp keeps the least key of its lanes (64-bit shuffles) and one atomicMin per warp folds it into keys[job].  The least
//            key is HM's first strict minimum in raster order (mvy outer, mvx inner); sad + cost < 2^23 + 2^16 never wraps.
//   prep     one thread per PU: decodes the key, writes (mv, sad) and completes the PU's sub-pel job (FRAC).
//   walk     one thread per FRAC PU: HM's 9-point half stage, then the 9-point quarter stage, over the 49-entry table.
// B(v) = xGetComponentBits, cost_s(x, y) = (uint32)(lambda * (B((x << s) - predX) + B((y << s) - predY))) >> 16: the 32-bit product
// wraps, as m_uiCost * getBits(x, y) >> 16 does in TComRdCost.
// =============================================================================================================================
constexpr unsigned long long kMeNoKey = ~0ull;
struct MeSearchCost {
  uint32_t lambda;     // m_uiCost = floor(65536 sqrt(lambda))
  int32_t predX, predY;  // m_mvPredictor in quarter pels
  int32_t frac;        // index of the PU's sub-pel job, -1 without CUCD_SEARCH_FRAC
};
struct MeArgmin { const MeSearchCost* cost; unsigned long long* keys; };   // the Argmin epilogue's inputs (null in the Surface form)
struct MeSearchOut { int32_t mvx, mvy; uint32_t sad; int32_t qmvx, qmvy; uint32_t fracCost; };   // = cucd_search_result
enum class MeOut { Surface, Argmin };

CUCD_HD int me_clz(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return __clz(v);
#else
  return __builtin_clz(v);
#endif
}
CUCD_HD uint32_t me_mv_bits(int v) {                     // xGetComponentBits: 1 + 2 floor(log2 t), t = v <= 0 ? -2v + 1 : 2v
  const uint32_t t = v <= 0 ? ((uint32_t)-v << 1) + 1u : (uint32_t)v << 1;
  return 1u + 2u * (uint32_t)(31 - me_clz(t));
}
CUCD_HD uint32_t me_mv_cost(const MeSearchCost& c, int x, int y, int s) {
  return (c.lambda * (me_mv_bits(x * (1 << s) - c.predX) + me_mv_bits(y * (1 << s) - c.predY))) >> 16;
}
// the key of candidate (dx, dy) of a cols-wide window whose top-left MV is (left, top)
CUCD_HD unsigned long long me_search_key(uint32_t sad, int dx, int dy, int cols, int left, int top, const MeSearchCost& c) {
  return ((unsigned long long)(sad + me_mv_cost(c, left + dx, top + dy, 2)) << 32) | (uint32_t)(dy * cols + dx);
}
CUCD_HD unsigned long long me_key_min(unsigned long long a, unsigned long long b) { return b < a ? b : a; }
// least key of a dy-lane thread's K candidates dx = dx0 + SPW k, dy (sad[] as the dy-lane SAD runs leave them, before the output shifts)
template <int K, int SPW>
CUCD_HD unsigned long long me_dy_lane_key(const uint32_t* sad, int subShift, int shiftOut, bool valid, int dx0, int dy, int cols, int left, int top,
                                          const MeSearchCost& c) {
  if (!valid) return kMeNoKey;
  // dx grows with i: the first strict minimum of sad + cost is the least key (32-bit compares keep the M tile's registers free)
  const uint32_t costY = me_mv_bits((top + dy) * 4 - c.predY);
  uint32_t best = 0xffffffffu;
  int bi = 0;
#pragma unroll
  for (int i = 0; i < K; i++) {
    const uint32_t v = ((sad[i] << subShift) >> shiftOut) + ((c.lambda * (me_mv_bits((left + dx0 + SPW * i) * 4 - c.predX) + costY)) >> 16);
    if (i == 0 || v < best) { best = v; bi = i; }
  }
  return ((unsigned long long)best << 32) | (uint32_t)(dy * cols + dx0 + SPW * bi);
}
#if defined(__CUDACC__)
// every lane of the warp takes part (lanes without a candidate bring kMeNoKey); lane 0 folds the warp's least key into *key
__device__ __forceinline__ void me_key_warp_commit(unsigned long long k, int lane, unsigned long long* key) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) k = me_key_min(k, __shfl_xor_sync(0xffffffffu, k, m));
  if (lane == 0 && k != kMeNoKey) atomicMin(key, k);
}
#endif

// prep, thread i < nPU: the integer result of PU i from its key; a FRAC PU's sub-pel job (pre-filled by the host with the PU origin
// in refOff) moves to the integer MV.  Job = MeJob, Sub = SubpelJob (kernels.h)
template <class Job, class Sub>
CUCD_HD void me_search_prep(int i, const unsigned long long* keys, const Job* jobs, const MeSearchCost* costs, const int32_t* refStride,
                            const Sub* subIn, Sub* subOut, MeSearchOut* out) {
  const Job& j = jobs[i];
  const MeSearchCost& c = costs[i];
  const unsigned long long k = keys[i];
  const int cols = j.right - j.left + 1;
  const uint32_t idx = (uint32_t)k, dy = idx / (uint32_t)cols, dx = idx - dy * (uint32_t)cols;
  const int mvx = j.left + (int)dx, mvy = j.top + (int)dy;
  MeSearchOut o;
  o.mvx = mvx; o.mvy = mvy; o.sad = (uint32_t)(k >> 32) - me_mv_cost(c, mvx, mvy, 2);
  o.qmvx = 4 * mvx; o.qmvy = 4 * mvy; o.fracCost = 0;
  out[i] = o;
  if (c.frac >= 0) {
    Sub sj = subIn[c.frac];
    sj.refOff += mvy * refStride[sj.refSlot] + mvx;
    subOut[c.frac] = sj;
  }
}

// walk: HM's orders of the half stage (s_acMvRefineH) and of the quarter stage (s_acMvRefineQ); each stage starts from the largest
// distortion and keeps the first strict minimum
CUCD_HD void me_search_walk(const uint32_t* T /*49*/, const MeSearchCost& c, MeSearchOut& o) {
  const int hx[9] = {0, 0, 0, -1, 1, -1, 1, -1, 1}, hy[9] = {0, -1, 1, 0, 0, -1, -1, 1, 1};
  const int qx[9] = {0, 0, 0, -1, 1, -1, 1, -1, 1}, qy[9] = {0, -1, 1, -1, -1, 0, 0, 1, 1};
  const int mvx = o.mvx, mvy = o.mvy;
  uint32_t best = 0xffffffffu;
  int bx = 0, by = 0;
  for (int i = 0; i < 9; i++) {
    const uint32_t d = T[(2 * hy[i] + 3) * 7 + 2 * hx[i] + 3] + me_mv_cost(c, 2 * mvx + hx[i], 2 * mvy + hy[i], 1);
    if (d < best) { best = d; bx = hx[i]; by = hy[i]; }
  }
  best = 0xffffffffu;
  int qbx = 0, qby = 0;
  for (int i = 0; i < 9; i++) {
    const uint32_t d = T[(2 * by + qy[i] + 3) * 7 + 2 * bx + qx[i] + 3] + me_mv_cost(c, 4 * mvx + 2 * bx + qx[i], 4 * mvy + 2 * by + qy[i], 0);
    if (d < best) { best = d; qbx = qx[i]; qby = qy[i]; }
  }
  o.qmvx = 4 * mvx + 2 * bx + qbx; o.qmvy = 4 * mvy + 2 * by + qby; o.fracCost = best;
}

// =============================================================================================================================
// TZ search (cucd_me_tz_search): the integer walk of xTZSearch with TZ_SEARCH_CONFIGURATION (TEncSearch.cpp: xTZSearch,
// xTZSearchHelp, xTZ8PointDiamondSearch, xTZ2PointSearch; include/cucudecide.h states the rules), then the refinement walk of
// cucd_me_search.  One warp per (PU, reference) job; a CTA takes up to kTzWarps jobs of one PU shape.
// The walk is a chain of STAGES whose centre is fixed while they run: the start points, the first search (the diamonds
// D = 1, 2, 4, .. <= search_range, stopped after three rounds without a better point), the two-point search, the raster and every
// star-refinement iteration.  A stage is a list of points in HM's order, cut into SEGMENTS (a diamond each; one segment for the
// two-point search and the raster; one per start point).  A segment's outcome is its least key (cost << 32 | point index), folded
// into the walk's state with one strict '<' (me_tz_fold): the same as HM's sequence of probes, because a point of a segment never
// sees the update of another point of the same segment (fixed centre) and a point visited again cannot beat the best.
//   lanes   G lanes (a power of two, me_tz_lanes) share one probe's samples, so a chunk of 32 / G consecutive points of the stage runs
//           at once; a group's partial sums meet through xor shuffles inside the group, a segment's keys through xor shuffles
//           across the groups.  Chunks run in order and stop once the first search's stop has been decided.
// =============================================================================================================================
constexpr int kTzWarps = 4;                    // jobs of a CTA
constexpr int kTz2Nx2N = 4;                    // CUCD_SEARCH_TZ_2NX2N
struct MeTzJob {
  int32_t curOff;                              // PU origin inside the current picture plane
  int32_t refOff;                              // co-located sample (mv 0) inside the padded plane of refSlot
  int32_t refSlot;
  int16_t w, h, subShift, flags;               // subShift: 0 for the generic widths (me_width_is_hm)
  int16_t left, right, top, bottom;            // the descriptor window `win`
  int16_t clipL, clipR, clipT, clipB;          // the clip box: every probe lies inside it
  int16_t mv2nX, mv2nY, range, pad;
  int32_t outIndex;                            // PU index in the caller's order (costs, results)
};
inline int me_tz_class(int w, int h) { return ((w >> 2) - 1) * 16 + (h >> 2) - 1; }
constexpr int kTzClasses = 16 * 16;
inline int me_tz_plan(int n, const MeTzJob* jobs, MeTzJob* sorted, int32_t* ctaFirst) {
  return me_plan_classes<kTzClasses>(n, jobs, sorted, ctaFirst, [](const MeTzJob& j) { return me_tz_class(j.w, j.h); }, [](const MeTzJob&) { return kTzWarps; });
}
// lanes per probe: about 16 samples per lane (an 8x8 PU: 4 lanes, 8 probes at once; 32x32 and up: one probe per warp)
CUCD_HD int me_tz_lanes(int samples) { int g = 1; while (g < 32 && 16 * g < samples) g <<= 1; return g; }

struct MeTzWin { int left, right, top, bottom; };
struct MeTzState { int bx, by; uint32_t best; int dist, round, pt; };
struct MeTzPoint { int x, y, p, d; bool ok; };
enum { kTzStart = 0, kTzDiamonds = 1, kTzTwo = 2, kTzRaster = 3 };
struct MeTzStage {
  int kind, cx, cy, n, stop;                   // n points; stop: the first search's three-round stop
  MeTzWin win;                                 // the guard window; the raster window for kTzRaster
  int pt, cols;                                // kTzTwo: the case; kTzRaster: points per row
  int sx0, sy0, sx2, sy2;                      // kTzStart: the predictor and the 2Nx2N start (point 1 is (0, 0))
};
CUCD_HD int me_tz_clamp(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
// first point of segment k (k = segment count: the stage's n)
CUCD_HD int me_tz_seg_first(const MeTzStage& s, int k) {
  if (s.kind == kTzStart) return k;
  if (s.kind != kTzDiamonds) return k ? s.n : 0;
  return k == 0 ? 0 : (k <= 4 ? 4 + 8 * (k - 1) : 28 + 16 * (k - 4));
}
CUCD_HD int me_tz_seg_of(const MeTzStage& s, int i) {
  if (s.kind == kTzStart) return i;
  if (s.kind != kTzDiamonds) return 0;
  return i < 4 ? 0 : (i < 28 ? 1 + ((i - 4) >> 3) : 4 + ((i - 28) >> 4));
}
// the diamonds D = 1, 2, 4, .. <= range around (cx, cy)
CUCD_HD MeTzStage me_tz_diamonds(int cx, int cy, const MeTzWin& win, int range, int stop) {
  MeTzStage s{};
  s.kind = kTzDiamonds; s.cx = cx; s.cy = cy; s.win = win; s.stop = stop;
  int k = 0;
  for (int D = 1; D <= range; D <<= 1) k++;
  s.n = me_tz_seg_first(s, k);
  return s;
}
CUCD_HD MeTzStage me_tz_two(int cx, int cy, const MeTzWin& win, int pt) {
  MeTzStage s{};
  s.kind = kTzTwo; s.cx = cx; s.cy = cy; s.win = win; s.pt = pt; s.n = pt >= 1 && pt <= 8 ? 2 : 0;
  return s;
}
CUCD_HD MeTzStage me_tz_raster(const MeTzWin& r) {
  MeTzStage s{};
  s.kind = kTzRaster; s.win = r; s.cols = (r.right - r.left) / 5 + 1; s.n = s.cols * ((r.bottom - r.top) / 5 + 1);
  return s;
}
// point i of a stage.  Guards: a point that moves left / right / up / down from the centre must not cross win's left / right / top /
// bottom border - xTZ8PointDiamondSearch's and xTZ2PointSearch's tests, which the all-inside branches pass anyway.
// Offsets are packed tables (no indexed local arrays in the kernel): a direction nibble is (sx + 1) | (sy + 1) << 2, sx, sy in -1..1.
CUCD_HD int me_tz_dir_x(uint32_t e) { return (int)(e & 3u) - 1; }
CUCD_HD int me_tz_dir_y(uint32_t e) { return (int)((e >> 2) & 3u) - 1; }
CUCD_HD MeTzPoint me_tz_point(const MeTzStage& s, int i) {
  MeTzPoint q;
  int dx = 0, dy = 0;
  q.p = 0;
  if (s.kind == kTzStart) {
    q.x = i == 0 ? s.sx0 : (i == 1 ? 0 : s.sx2); q.y = i == 0 ? s.sy0 : (i == 1 ? 0 : s.sy2); q.d = 0; q.ok = true;
    return q;
  }
  if (s.kind == kTzRaster) {
    const int r = i / s.cols;
    q.x = s.win.left + 5 * (i - r * s.cols); q.y = s.win.top + 5 * r; q.d = 5; q.ok = true;
    return q;
  }
  if (s.kind == kTzTwo) {
    // xTZ2PointSearch, cases 1..8: byte pt - 1 holds the first point's direction in its low nibble, the second's in its high nibble
    const uint32_t e = (uint32_t)(0x96A894A208612014ull >> (8 * (s.pt - 1) + 4 * i)) & 15u;
    dx = me_tz_dir_x(e); dy = me_tz_dir_y(e); q.d = 2;
  } else {
    const int k = me_tz_seg_of(s, i), D = 1 << k, j = i - me_tz_seg_first(s, k);
    q.d = D;
    if (D <= 8) {
      // D = 1: up, left, right, down (points 2, 4, 5, 7); D = 2..8: up, the two upper diagonals, left, right, the two lower diagonals,
      // down (points 2, 1, 3, 4, 5, 6, 8, 7), the diagonals at D / 2
      const uint32_t e = D == 1 ? (0x9641u >> (4 * j)) & 15u : (0x9A864201u >> (4 * j)) & 15u;
      q.p = (int)(((D == 1 ? 0x7542u : 0x78654312u) >> (4 * j)) & 15u);
      const int sx = me_tz_dir_x(e), sy = me_tz_dir_y(e), a = (sx != 0 && sy != 0) ? D >> 1 : D;
      dx = sx * a; dy = sy * a;
      if (sx != 0 && sy != 0) q.d = D >> 1;
    } else if (j < 4) {
      const uint32_t e = (0x9641u >> (4 * j)) & 15u;                  // up, left, right, down
      dx = me_tz_dir_x(e) * D; dy = me_tz_dir_y(e) * D;
    } else {
      const int qk = (D >> 2) * (((j - 4) >> 2) + 1), m = (j - 4) & 3;  // k = 1..3: upper left, upper right, lower left, lower right
      dx = (m & 1) ? qk : -qk; dy = (m & 2) ? D - qk : qk - D;
    }
  }
  q.x = s.cx + dx; q.y = s.cy + dy;
  q.ok = (dx >= 0 || q.x >= s.win.left) && (dx <= 0 || q.x <= s.win.right) && (dy >= 0 || q.y >= s.win.top) && (dy <= 0 || q.y <= s.win.bottom);
  return q;
}
// segment k's least key has been found: HM's round count, then one strict '<'.  Returns true when the stage stops here.
CUCD_HD bool me_tz_fold(MeTzState& st, const MeTzStage& s, unsigned long long key) {
  if (s.kind == kTzDiamonds) st.round++;
  if (key != kMeNoKey && (uint32_t)(key >> 32) < st.best) {
    const MeTzPoint q = me_tz_point(s, (int)(uint32_t)key);
    st.best = (uint32_t)(key >> 32); st.bx = q.x; st.by = q.y; st.dist = q.d; st.round = 0; st.pt = q.p;
  }
  return s.stop && st.round >= 3;
}
// xTZSearch's sequence of stages.  run(stage, state) evaluates a stage and folds its segments into the state (the kernel: a warp,
// the CPU replay: 32 emulated lanes); the clip box bounds the start points, win guards the diamonds and the two-point search.
template <class Run>
CUCD_HD MeTzState me_tz_walk(const MeTzJob& j, const MeSearchCost& c, Run&& run) {
  MeTzState st;
  st.bx = 0; st.by = 0; st.best = 0xffffffffu; st.dist = 0; st.round = 0; st.pt = 0;
  const MeTzWin win{j.left, j.right, j.top, j.bottom};
  MeTzStage s{};
  s.kind = kTzStart; s.n = (j.flags & kTz2Nx2N) ? 3 : 2;
  s.sx0 = me_tz_clamp(c.predX, 4 * j.clipL, 4 * j.clipR) >> 2; s.sy0 = me_tz_clamp(c.predY, 4 * j.clipT, 4 * j.clipB) >> 2;
  s.sx2 = me_tz_clamp(j.mv2nX, j.clipL, j.clipR); s.sy2 = me_tz_clamp(j.mv2nY, j.clipT, j.clipB);
  run(s, st);
  MeTzWin rwin = win;                                                   // xSetSearchRange around the best start (TZ_2NX2N)
  if (j.flags & kTz2Nx2N)
    rwin = MeTzWin{me_tz_clamp(st.bx - j.range, j.clipL, j.clipR), me_tz_clamp(st.bx + j.range, j.clipL, j.clipR),
                   me_tz_clamp(st.by - j.range, j.clipT, j.clipB), me_tz_clamp(st.by + j.range, j.clipT, j.clipB)};
  run(me_tz_diamonds(st.bx, st.by, win, j.range, 1), st);
  if (st.dist == 1) { st.dist = 0; run(me_tz_two(st.bx, st.by, win, st.pt), st); }
  if (st.dist > 5) { st.dist = 5; run(me_tz_raster(rwin), st); }
  while (st.dist > 0) {                                                 // ends: every iteration that goes on lowered best
    const int cx = st.bx, cy = st.by;
    st.dist = 0; st.pt = 0;
    run(me_tz_diamonds(cx, cy, win, j.range, 0), st);
    if (st.dist == 1) { st.dist = 0; if (st.pt != 0) run(me_tz_two(st.bx, st.by, win, st.pt), st); }
  }
  return st;
}
CUCD_HD int16_t me_ld16(const int16_t* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}
// lane g of the G lanes that probe the reference block at ref: its part of sum |cur - ref| over the staged rows (nr rows of w samples,
// row r of the PU at r << subShift); sample index s = r w + col, s / w as one multiply-high (s w < 2^32)
CUCD_HD uint32_t me_tz_sad_part(const int16_t* sCur, const int16_t* ref, int refStride, int w, int nr, int subShift, int g, int G) {
  const uint32_t invW = me_inv((uint32_t)w);
  uint32_t acc = 0;
  for (int s = g; s < nr * w; s += G) {
    const int r = (int)me_mulhi((uint32_t)s, invW), col = s - r * w;
    acc += (uint32_t)iabs32((int)sCur[s] - (int)me_ld16(ref + (long long)(r << subShift) * refStride + col));
  }
  return acc;
}
// the probe's value c = SAD + cost_2 from the group's total (xGetSAD*: << iSubShift, then >> (bitDepth - 8))
CUCD_HD uint32_t me_tz_probe_cost(uint32_t total, int subShift, int bitDepth, const MeSearchCost& c, int x, int y) {
  return ((total << subShift) >> (bitDepth - 8)) + me_mv_cost(c, x, y, 2);
}
// the integer result of a finished walk, and the PU's sub-pel job (FRAC) moved to it; Sub = SubpelJob (kernels.h)
template <class Sub>
CUCD_HD void me_tz_finish(const MeTzState& st, const MeTzJob& j, const MeSearchCost& c, int refStride, const Sub* subIn, Sub* subOut, MeSearchOut* out) {
  MeSearchOut o;
  o.mvx = st.bx; o.mvy = st.by; o.sad = st.best - me_mv_cost(c, st.bx, st.by, 2);
  o.qmvx = 4 * st.bx; o.qmvy = 4 * st.by; o.fracCost = 0;
  out[j.outIndex] = o;
  if (c.frac >= 0) {
    Sub sj = subIn[c.frac];
    sj.refOff += st.by * refStride + st.bx;
    subOut[c.frac] = sj;
  }
}

}  // namespace cucd
