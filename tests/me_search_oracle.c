/* me_search_oracle.c - CPU restatement of HM's full-search motion estimation and its sub-pel refinement walk (TEST INFRASTRUCTURE:
 * the checker of cucd_me_search; the product never links it).  Built by tests/me_search_util.py load_me_search_oracle() into one
 * library with oracle/cucd_oracle.c.  It adds no distortion arithmetic of its own: the SADs are oracle_sad_surface's, the 49-point
 * table is oracle_subpel_surface's (both pinned against encoder dumps by tests/golden); this file adds the motion-vector cost and the
 * two minimum rules on top.
 *
 * Parity status: the orders and formulas below restate HM-16.3; they are NOT pinned against the reference sources, which are not part
 * of this repository.  tests/test_me_search_oracle.py pins them against an independent numpy statement.
 *
 * Reference lines (HM-16.3):
 *   TComRdCost.h  xGetComponentBits     uiLength = 1, uiTemp = v <= 0 ? (-v << 1) + 1 : v << 1; while (uiTemp != 1) { uiTemp >>= 1;
 *                                       uiLength += 2; }
 *   TComRdCost.h  getCost(x, y)         m_uiCost * getBits(x, y) >> 16, getBits = B((x << m_iCostScale) - m_mvPredictor.hor) + B(..)
 *   TEncSearch.cpp:3886-3943            xPatternSearch: for y = top..bottom, for x = left..right: uiSad = DistFunc + getCost(x, y)
 *                                       (cost scale 2); uiSad < uiSadBest keeps the first strict minimum
 *   TEncSearch.cpp:808-865              xPatternRefinement: uiDistBest = MAX; for the 9 points of the stage: uiDist = DistFunc +
 *                                       getCost(cMvTest) with cMvTest = pcMvRefine[i] + baseRefMv << (2 - uiFrac);
 *                                       uiDist < uiDistBest; rcMvFrac = pcMvRefine[uiDirecBest]
 *   TEncSearch.cpp:4340-4376            xPatternSearchFracDIF: half stage (cost scale 1, s_acMvRefineH), then quarter stage around
 *                                       the half result (cost scale 0, s_acMvRefineQ); ruiCost = the quarter stage's best
 */
#include <stdint.h>
#include <stdlib.h>
#include "cucd_oracle.h"

/* xGetComponentBits, the loop form */
uint32_t oracle_mv_bits(int v) {
  uint32_t len = 1, t = v <= 0 ? ((uint32_t)(-(int64_t)v) << 1) + 1u : (uint32_t)v << 1;
  while (t != 1) { t >>= 1; len += 2; }
  return len;
}

/* getCost of the mv (x, y) at cost scale s: the 32-bit unsigned product wraps */
uint32_t oracle_mv_cost(uint32_t lambda, int x, int y, int s, int predX, int predY) {
  return (uint32_t)(lambda * (oracle_mv_bits(x * (1 << s) - predX) + oracle_mv_bits(y * (1 << s) - predY))) >> 16;
}

static const int kRefineH[9][2] = {{0, 0}, {0, -1}, {0, 1}, {-1, 0}, {1, 0}, {-1, -1}, {1, -1}, {-1, 1}, {1, 1}};
static const int kRefineQ[9][2] = {{0, 0}, {0, -1}, {0, 1}, {-1, -1}, {1, -1}, {-1, 0}, {1, 0}, {-1, 1}, {1, 1}};

/* the two 9-point stages over T[(dy + 3) * 7 + dx + 3] (quarter-pel offsets around the integer mv); qmv[2] the final quarter-pel MV */
void oracle_me_frac_walk(const uint32_t* T, int mvx, int mvy, int predX, int predY, uint32_t lambda, int32_t* qmv, uint32_t* fracCost) {
  uint32_t best = 0xffffffffu;
  int hb = 0, qb = 0, i;
  for (i = 0; i < 9; i++) {
    const int hx = kRefineH[i][0], hy = kRefineH[i][1];
    const uint32_t d = T[(2 * hy + 3) * 7 + 2 * hx + 3] + oracle_mv_cost(lambda, 2 * mvx + hx, 2 * mvy + hy, 1, predX, predY);
    if (d < best) { best = d; hb = i; }
  }
  const int bx = kRefineH[hb][0], by = kRefineH[hb][1];
  best = 0xffffffffu;
  for (i = 0; i < 9; i++) {
    const int qx = kRefineQ[i][0], qy = kRefineQ[i][1];
    const uint32_t d = T[(2 * by + qy + 3) * 7 + 2 * bx + qx + 3] + oracle_mv_cost(lambda, 4 * mvx + 2 * bx + qx, 4 * mvy + 2 * by + qy, 0, predX, predY);
    if (d < best) { best = d; qb = i; }
  }
  qmv[0] = 4 * mvx + 2 * bx + kRefineQ[qb][0];
  qmv[1] = 4 * mvy + 2 * by + kRefineQ[qb][1];
  *fracCost = best;
}

/* one PU: xPatternSearch over the inclusive window, then (flags & 1) the refinement walk with (flags & 2) Hadamard.
 * res[6] = mvx, mvy, sad, qmvx, qmvy, frac_cost (cucd_search_result).  Returns 0, or -1 when the surface cannot be allocated. */
int oracle_me_search(int bitDepth, const int16_t* org, int orgStride, int w, int h, const int16_t* refAtZeroMv, int refStride, int left, int right,
                     int top, int bottom, int subShift, int predX, int predY, uint32_t lambda, int flags, int32_t* res) {
  const int cols = right - left + 1, rows = bottom - top + 1;
  uint32_t* sad = (uint32_t*)malloc(sizeof(uint32_t) * (size_t)cols * rows);
  uint32_t best = 0xffffffffu, bestSad = 0;
  int bx = left, by = top, x, y;
  if (!sad) return -1;
  oracle_sad_surface(bitDepth, org, orgStride, w, h, refAtZeroMv, refStride, left, right, top, bottom, subShift, sad);
  for (y = top; y <= bottom; y++)
    for (x = left; x <= right; x++) {
      const uint32_t s = sad[(size_t)(y - top) * cols + (x - left)];
      const uint32_t c = s + oracle_mv_cost(lambda, x, y, 2, predX, predY);
      if (c < best) { best = c; bestSad = s; bx = x; by = y; }
    }
  free(sad);
  res[0] = bx; res[1] = by; res[2] = (int32_t)bestSad; res[3] = 4 * bx; res[4] = 4 * by; res[5] = 0;
  if (flags & 1) {
    uint32_t T[49], fc;
    int32_t qmv[2];
    oracle_subpel_surface(bitDepth, org, orgStride, w, h, refAtZeroMv, refStride, bx, by, (flags & 2) ? 1 : 0, T);
    oracle_me_frac_walk(T, bx, by, predX, predY, lambda, qmv, &fc);
    res[3] = qmv[0]; res[4] = qmv[1]; res[5] = (int32_t)fc;
  }
  return 0;
}
