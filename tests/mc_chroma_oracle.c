/* mc_chroma_oracle.c - CPU restatement of HM's 4:2:0 chroma motion compensation and chroma SSE of uni- and bi-predictive inter
 * candidates (TEST INFRASTRUCTURE: the checker of cucd_me_mc_chroma; the product never links it).  Built by
 * tests/mc_chroma_util.py load_mc_chroma_oracle() into one library with oracle/cucd_oracle.c, whose oracle_sse it uses.
 *
 * Parity status: NOT pinned against the reference's compiled functions or new encoder dumps (the reference sources are needed for
 * both).  It is written branch by branch from TComInterpolationFilter::filterCopy / filter<4, ...> with m_chromaFilter and the chroma
 * branch of TComPrediction::xPredInterBlk, plus TComYuv::addAvg, and tests/test_mc_chroma_oracle.py pins it in other ways: an
 * independent numpy statement of the same branches, integer MVs copy the reference, constant planes, bi with identical motion ==
 * uni, mirror symmetry of the half-sample filter, and sse == oracle_sse of the returned prediction.
 *
 * Reference symbols (HM-16.x):
 *   TComInterpolationFilter::m_chromaFilter     the eight 4-tap filters below, indexed by the eighth-pel fraction
 *   TComInterpolationFilter::filterCopy         isFirst == isLast: copy; isFirst: (src << shift) - IF_INTERNAL_OFFS; isLast:
 *                                               clip((src + IF_INTERNAL_OFFS + round) >> shift), shift = max(2, 14 - bitDepth)
 *   TComInterpolationFilter::filter<4, ...>     the shift / offset rules of filter4 below; filterHor / filterVer pick filterCopy at
 *                                               fraction 0
 *   TComPrediction::xPredInterBlk (chroma)      yFrac == 0 -> filterHor(xFrac, !bi); xFrac == 0 -> filterVer(yFrac, isFirst, !bi);
 *                                               else filterHor(xFrac, isLast = false) on h + 3 rows from ref - stride, then
 *                                               filterVer(yFrac, !isFirst, !bi) from tmp + one row
 *   TComYuv::addAvg                             clip((p0 + p1 + offset) >> shiftNum), shiftNum = max(2, 14 - bd) + 1,
 *                                               offset = (1 << (shiftNum - 1)) + 2 * IF_INTERNAL_OFFS
 *   TEncSearch::encodeResAndCalcRdInterCU       getDistPart of each chroma plane: TComRdCost::xGetSSE, before m_distortionWeight
 */
#include <stdint.h>
#include <string.h>
#include "cucd_oracle.h"

#define IF_INTERNAL_PREC 14
#define IF_FILTER_PREC 6
#define IF_INTERNAL_OFFS (1 << (IF_INTERNAL_PREC - 1))

static const int kChromaTaps[8][4] = {{0, 64, 0, 0},     {-2, 58, 10, -2}, {-4, 54, 16, -2}, {-6, 46, 28, -4},
                                      {-4, 36, 36, -4},  {-4, 28, 46, -6}, {-2, 16, 54, -4}, {-2, 10, 58, -2}};

static int imax(int a, int b) { return a > b ? a : b; }

/* filterCopy<isFirst, isLast> */
static void filter_copy(int bitDepth, const int16_t* src, int srcStride, int16_t* dst, int dstStride, int w, int h, int isFirst, int isLast) {
  const int shift = imax(2, IF_INTERNAL_PREC - bitDepth), maxVal = (1 << bitDepth) - 1;
  int r, c;
  for (r = 0; r < h; r++) for (c = 0; c < w; c++) {
    const int s = src[r * srcStride + c];
    int v;
    if (isFirst == isLast) v = s;
    else if (isFirst) v = (s << shift) - IF_INTERNAL_OFFS;
    else {
      v = (s + IF_INTERNAL_OFFS + (1 << (shift - 1))) >> shift;
      v = v < 0 ? 0 : (v > maxVal ? maxVal : v);
    }
    dst[r * dstStride + c] = (int16_t)v;
  }
}

/* filter<4, isVertical, isFirst, isLast>: src points at the sample the block's first output sits on; taps at -1 .. 2 */
static void filter4(int bitDepth, const int16_t* src, int srcStride, int16_t* dst, int dstStride, int w, int h, int frac, int isVertical, int isFirst,
                    int isLast) {
  const int headRoom = IF_INTERNAL_PREC - bitDepth, cStride = isVertical ? srcStride : 1, maxVal = (1 << bitDepth) - 1;
  int shift = IF_FILTER_PREC, offset, r, c, k;
  if (isLast) {
    shift += isFirst ? 0 : headRoom;
    offset = 1 << (shift - 1);
    offset += isFirst ? 0 : IF_INTERNAL_OFFS << IF_FILTER_PREC;
  } else {
    shift -= isFirst ? headRoom : 0;
    offset = isFirst ? -IF_INTERNAL_OFFS * (1 << shift) : 0;
  }
  for (r = 0; r < h; r++) for (c = 0; c < w; c++) {
    const int16_t* s = src + r * srcStride + c - cStride;
    int sum = 0, v;
    for (k = 0; k < 4; k++) sum += s[k * cStride] * kChromaTaps[frac][k];
    v = (sum + offset) >> shift;
    if (isLast) v = v < 0 ? 0 : (v > maxVal ? maxVal : v);
    dst[r * dstStride + c] = (int16_t)v;
  }
}

static void filter_hor(int bd, const int16_t* src, int ss, int16_t* dst, int ds, int w, int h, int frac, int isLast) {
  if (frac == 0) filter_copy(bd, src, ss, dst, ds, w, h, 1, isLast);
  else filter4(bd, src, ss, dst, ds, w, h, frac, 0, 1, isLast);
}
static void filter_ver(int bd, const int16_t* src, int ss, int16_t* dst, int ds, int w, int h, int frac, int isFirst, int isLast) {
  if (frac == 0) filter_copy(bd, src, ss, dst, ds, w, h, isFirst, isLast);
  else filter4(bd, src, ss, dst, ds, w, h, frac, 1, isFirst, isLast);
}

/* xPredInterBlk (chroma) of one list: bi = 0 -> the clipped prediction, bi = 1 -> the 14-bit intermediate.  ref: the block's
 * top-left at the INTEGER part of the eighth-pel MV; fx, fy = mv & 7 */
void oracle_interp_chroma(int bitDepth, const int16_t* ref, int stride, int w, int h, int fx, int fy, int bi, int16_t* out) {
  int16_t tmp[(32 + 3) * 32];
  if (fy == 0) filter_hor(bitDepth, ref, stride, out, w, w, h, fx, !bi);
  else if (fx == 0) filter_ver(bitDepth, ref, stride, out, w, w, h, fy, 1, !bi);
  else {
    filter_hor(bitDepth, ref - stride, stride, tmp, w, w, h + 3, fx, 0);
    filter_ver(bitDepth, tmp + w, w, out, w, w, h, fy, 0, !bi);
  }
}

/* motionCompensation's prediction of one chroma plane of a candidate: nl = 1 -> xPredInterUni; nl = 2 -> xPredInterBi: both lists at
 * 14 bits, then addAvg */
void oracle_mc_chroma_pred(int bitDepth, int nl, const int16_t* ref0, int stride0, int fx0, int fy0, const int16_t* ref1, int stride1, int fx1,
                           int fy1, int w, int h, int16_t* pred) {
  int16_t p0[32 * 32], p1[32 * 32];
  const int shiftNum = imax(2, IF_INTERNAL_PREC - bitDepth) + 1, offset = (1 << (shiftNum - 1)) + 2 * IF_INTERNAL_OFFS, maxVal = (1 << bitDepth) - 1;
  int i;
  if (nl == 1) { oracle_interp_chroma(bitDepth, ref0, stride0, w, h, fx0, fy0, 0, pred); return; }
  oracle_interp_chroma(bitDepth, ref0, stride0, w, h, fx0, fy0, 1, p0);
  oracle_interp_chroma(bitDepth, ref1, stride1, w, h, fx1, fy1, 1, p1);
  for (i = 0; i < w * h; i++) {
    int v = (p0[i] + p1[i] + offset) >> shiftNum;
    pred[i] = (int16_t)(v < 0 ? 0 : (v > maxVal ? maxVal : v));
  }
}

/* getDistPart of the chroma prediction (also written to pred when not NULL) against org */
uint32_t oracle_mc_chroma_cost(int bitDepth, const int16_t* org, int orgStride, int nl, const int16_t* ref0, int stride0, int fx0, int fy0,
                               const int16_t* ref1, int stride1, int fx1, int fy1, int w, int h, int16_t* pred) {
  int16_t p[32 * 32];
  oracle_mc_chroma_pred(bitDepth, nl, ref0, stride0, fx0, fy0, ref1, stride1, fx1, fy1, w, h, p);
  if (pred) memcpy(pred, p, sizeof(int16_t) * (size_t)w * h);
  return oracle_sse(bitDepth, org, orgStride, p, w, w, h);
}
