/* inter_tu_oracle.c - checker of the inter TU chain (cucd_inter_tu_*): the per-TU arithmetic of TEncSearch::xEstimateResidualQT
 * composed from the oracle's pinned functions.  The only new statement here is the order of the calls:
 *   nonCoeffDist = getDistPart(0, resi)                                  (the distortion of the TU coded with CBF 0)
 *   transformNxN: xT with useDST = 0 (TComTU::useDST is intra-only) or xTransformSkip
 *   xQuant: flat scaling, offset 85/512 (an inter CU never lies in an I slice), signBitHidingHDQ on the diagonal scan
 *           (getCoefScanIdx of a non-intra CU)
 *   invTransformNxN: xDeQuant + xIT (useDST = 0) or xITransformSkip; rresi = 0 when every level is zero
 *   dist = getDistPart(rresi, resi)                                      (TComRdCost.cpp:433-455, uint32 with wrap-around)
 * Chroma blocks take the same path (4:2:0: DCT, diagonal scan); their distortion is returned before m_distortionWeight. */
#include <stdint.h>
#include <string.h>
#include "cucd_oracle.h"

/* stage 0: coef (and distZero) only; 1: the whole chain with the plain quantiser (level out); 2: from GIVEN levels (level in).
 * resi: n x n residual with row stride `stride`; coef / level / rresi: n*n row-major.  coef, rresi, distZero, absSum may be NULL. */
void oracle_inter_tu(int bitDepth, int n, int qp, int transformSkip, int chroma, int signHiding, int stage, const int16_t* resi, int stride,
                     int32_t* coef, int32_t* level, int16_t* rresi, uint32_t* dist, uint32_t* distZero, int32_t* absSum) {
  static const int16_t zeros[32 * 32];
  int16_t r[32 * 32];
  int32_t c[32 * 32], deq[32 * 32];
  int i, sum = 0;
  (void)chroma;                                                          /* 4:2:0 chroma: the same transform and scan as luma */
  if (distZero) *distZero = oracle_sse(bitDepth, resi, stride, zeros, n, n, n);
  if (stage != 2) {
    if (transformSkip) oracle_transform_skip(bitDepth, n, resi, stride, c); else oracle_fwd_transform(bitDepth, n, 0, resi, stride, c);
    if (coef) memcpy(coef, c, (size_t)n * n * sizeof(int32_t));
    if (stage == 0) return;
    sum = oracle_quant(bitDepth, n, qp, 0, signHiding, 0, c, level);
  } else {
    for (i = 0; i < n * n; i++) sum += level[i] < 0 ? -level[i] : level[i];   /* only its being non-zero matters */
  }
  if (absSum) *absSum = sum;
  if (sum > 0) {
    oracle_dequant(bitDepth, n, qp, level, deq);
    if (transformSkip) oracle_inv_transform_skip(bitDepth, n, deq, r, n); else oracle_inv_transform(bitDepth, n, 0, deq, r, n);
  } else {
    if (stage == 1) memset(level, 0, (size_t)n * n * sizeof(int32_t));
    memset(r, 0, sizeof(r));
  }
  if (rresi) memcpy(rresi, r, (size_t)n * n * sizeof(int16_t));
  *dist = oracle_sse(bitDepth, resi, stride, r, n, n, n);
}
