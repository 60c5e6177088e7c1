/* mc_oracle.c - CPU restatement of HM's luma motion compensation for uni- and bi-predictive inter candidates (TEST
 * INFRASTRUCTURE: the checker of cucd_me_mc_cost; the product never links it).  Built by tests/_util.py load_mc_oracle() into one
 * library with oracle/cucd_oracle.c, whose oracle_interp_luma / oracle_satd it uses.
 *
 * Parity status: NOT pinned against the reference's compiled functions or new encoder dumps (the reference sources are needed for
 * both).  It is written branch by branch from TComInterpolationFilter::filter / filterCopy and TComPrediction::xPredInterBlk, and the
 * tests pin it in other ways: an independent numpy statement of the same branches, constant planes, bi with identical motion ==
 * uni (what xCheckIdenticalMotion relies on), and uni costs == oracle_subpel_surface entries, which tests/golden/frac_*.npz pin.
 *
 * Reference lines (HM-16.x):
 *   TComInterpolationFilter.cpp:57-63   luma taps
 *   TComInterpolationFilter.cpp:83-133  filterCopy<isFirst, isLast>: copy / (src << shift) - IF_INTERNAL_OFFS /
 *                                       clip((src + IF_INTERNAL_OFFS + round) >> shift), shift = max(2, 14 - bitDepth)
 *   TComInterpolationFilter.cpp:150-290 filter<N, isVertical, isFirst, isLast>: shift / offset rules below
 *   TComPrediction.cpp:560-600          xPredInterBlk luma: yFrac == 0 -> filterHor(xFrac, !bi); xFrac == 0 -> filterVer(yFrac, isFirst,
 *                                       !bi); else filterHor(xFrac, isLast = false) on h + 7 rows, filterVer(yFrac, !isFirst, !bi)
 *   TComYuv.cpp:260-310                 addAvg: clip((p0 + p1 + offset) >> shiftNum), shiftNum = max(2, 14 - bd) + 1,
 *                                       offset = (1 << (shiftNum - 1)) + 2 * IF_INTERNAL_OFFS
 *   TEncSearch.cpp:2905-2926            xGetInterPredictionError: DistFunc of the luma prediction, HADME -> xGetHADs, else xGetSAD,
 *                                       iSubShift 0
 */
#include <stdint.h>
#include <string.h>
#include "cucd_oracle.h"

#define IF_INTERNAL_PREC 14
#define IF_FILTER_PREC 6
#define IF_INTERNAL_OFFS (1 << (IF_INTERNAL_PREC - 1))

static const int kTaps[4][8] = {{0, 0, 0, 64, 0, 0, 0, 0}, {-1, 4, -10, 58, 17, -5, 1, 0}, {-1, 4, -11, 40, 40, -11, 4, -1}, {0, 1, -5, 17, 58, -10, 4, -1}};

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

/* filter<8, isVertical, isFirst, isLast>: src points at the sample the block's first output sits on */
static void filter8(int bitDepth, const int16_t* src, int srcStride, int16_t* dst, int dstStride, int w, int h, int frac, int isVertical, int isFirst,
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
    const int16_t* s = src + r * srcStride + c - 3 * cStride;
    int sum = 0, v;
    for (k = 0; k < 8; k++) sum += s[k * cStride] * kTaps[frac][k];
    v = (sum + offset) >> shift;
    if (isLast) v = v < 0 ? 0 : (v > maxVal ? maxVal : v);
    dst[r * dstStride + c] = (int16_t)v;
  }
}

static void filter_hor(int bd, const int16_t* src, int ss, int16_t* dst, int ds, int w, int h, int frac, int isLast) {
  if (frac == 0) filter_copy(bd, src, ss, dst, ds, w, h, 1, isLast);
  else filter8(bd, src, ss, dst, ds, w, h, frac, 0, 1, isLast);
}
static void filter_ver(int bd, const int16_t* src, int ss, int16_t* dst, int ds, int w, int h, int frac, int isFirst, int isLast) {
  if (frac == 0) filter_copy(bd, src, ss, dst, ds, w, h, isFirst, isLast);
  else filter8(bd, src, ss, dst, ds, w, h, frac, 1, isFirst, isLast);
}

/* xPredInterBlk (luma) with bi = true: the 14-bit intermediate of one list.  ref: the block's top-left at the INTEGER part of the MV */
void oracle_interp_luma14(int bitDepth, const int16_t* ref, int stride, int w, int h, int fx, int fy, int16_t* out) {
  int16_t tmp[(64 + 7) * 64];
  if (fy == 0) filter_hor(bitDepth, ref, stride, out, w, w, h, fx, 0);
  else if (fx == 0) filter_ver(bitDepth, ref, stride, out, w, w, h, fy, 1, 0);
  else {
    filter_hor(bitDepth, ref - 3 * stride, stride, tmp, w, w, h + 7, fx, 0);
    filter_ver(bitDepth, tmp + 3 * w, w, out, w, w, h, fy, 0, 0);
  }
}

/* motionCompensation's luma prediction of one candidate: nl = 1 -> xPredInterUni (oracle_interp_luma, pinned by frac_*.npz);
 * nl = 2 -> xPredInterBi: both lists at 14 bits, then addAvg */
void oracle_mc_pred(int bitDepth, int nl, const int16_t* ref0, int stride0, int fx0, int fy0, const int16_t* ref1, int stride1, int fx1, int fy1,
                    int w, int h, int16_t* pred) {
  int16_t p0[64 * 64], p1[64 * 64];
  const int shiftNum = imax(2, IF_INTERNAL_PREC - bitDepth) + 1, offset = (1 << (shiftNum - 1)) + 2 * IF_INTERNAL_OFFS, maxVal = (1 << bitDepth) - 1;
  int i;
  if (nl == 1) { oracle_interp_luma(bitDepth, ref0, stride0, w, h, fx0, fy0, pred); return; }
  oracle_interp_luma14(bitDepth, ref0, stride0, w, h, fx0, fy0, p0);
  oracle_interp_luma14(bitDepth, ref1, stride1, w, h, fx1, fy1, p1);
  for (i = 0; i < w * h; i++) {
    int v = (p0[i] + p1[i] + offset) >> shiftNum;
    pred[i] = (int16_t)(v < 0 ? 0 : (v > maxVal ? maxVal : v));
  }
}

/* xGetInterPredictionError on the luma block: the prediction (also written to pred when not NULL) against org */
uint32_t oracle_mc_cost(int bitDepth, const int16_t* org, int orgStride, int nl, const int16_t* ref0, int stride0, int fx0, int fy0, const int16_t* ref1,
                        int stride1, int fx1, int fy1, int w, int h, int useHadamard, int16_t* pred) {
  int16_t p[64 * 64];
  oracle_mc_pred(bitDepth, nl, ref0, stride0, fx0, fy0, ref1, stride1, fx1, fy1, w, h, p);
  if (pred) memcpy(pred, p, sizeof(int16_t) * (size_t)w * h);
  if (useHadamard) return oracle_satd(bitDepth, org, orgStride, p, w, w, h);
  return oracle_sad(bitDepth, org, orgStride, p, w, w, h, 0);
}
