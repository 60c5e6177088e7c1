/* me_tz_oracle.c - CPU restatement of HM's TZ search (TEST INFRASTRUCTURE: the checker of cucd_me_tz_search; the product never links
 * it).  Built by tests/me_tz_util.py load_me_tz_oracle() into one library with oracle/cucd_oracle.c and tests/me_search_oracle.c.  It
 * adds only the walk: the SADs are oracle_sad_surface's (1x1 windows, or a caller-given surface), the motion-vector cost is
 * oracle_mv_cost and the refinement is oracle_subpel_surface + oracle_me_frac_walk.
 *
 * Parity status: the walk below restates HM-16.3 TEncSearch.cpp xTZSearch / xTZSearchHelp / xTZ8PointDiamondSearch / xTZ2PointSearch
 * with TZ_SEARCH_CONFIGURATION (iRaster 5, zero-vector test, first search diamond stopped after 3 rounds, raster on, raster
 * refinement off, star refinement diamond without stop); it is NOT pinned against the reference sources, which are not part of this
 * repository.  tests/test_me_tz_oracle.py pins it against an independent Python statement.
 * The walk is written the way HM writes it: probe by probe, with the all-inside branch of the diamond and the per-border branch.
 */
#include <stdint.h>
#include <stdlib.h>
#include "cucd_oracle.h"

uint32_t oracle_mv_cost(uint32_t lambda, int x, int y, int s, int predX, int predY);
void oracle_me_frac_walk(const uint32_t* T, int mvx, int mvy, int predX, int predY, uint32_t lambda, int32_t* qmv, uint32_t* fracCost);

typedef struct {
  int bitDepth, orgStride, w, h, refStride, subShift;
  const int16_t* org;
  const int16_t* ref;
  const uint32_t* surf;
  int sl, sr, st, sb;
  uint32_t lambda;
  int predX, predY;
  int left, right, top, bottom;      /* win */
  int bx, by, dist, round, pt;
  uint32_t best;
  int32_t* trace;
  int cap, n, stage, err;
} Tz;

/* xTZSearchHelp */
static void probe(Tz* t, int x, int y, int p, int d) {
  uint32_t sad = 0, c;
  if (t->surf) {
    if (x < t->sl || x > t->sr || y < t->st || y > t->sb) { t->err = 1; return; }
    sad = t->surf[(size_t)(y - t->st) * (t->sr - t->sl + 1) + (x - t->sl)];
  } else {
    oracle_sad_surface(t->bitDepth, t->org, t->orgStride, t->w, t->h, t->ref, t->refStride, x, x, y, y, t->subShift, &sad);
  }
  c = sad + oracle_mv_cost(t->lambda, x, y, 2, t->predX, t->predY);
  if (t->trace && t->n < t->cap) {
    int32_t* e = t->trace + 6 * t->n;
    e[0] = x; e[1] = y; e[2] = p; e[3] = d; e[4] = t->stage; e[5] = (int32_t)c;
  }
  t->n++;
  if (c < t->best) { t->best = c; t->bx = x; t->by = y; t->dist = d; t->round = 0; t->pt = p; }
}

/* xTZ8PointDiamondSearch */
static void diamond(Tz* t, int cx, int cy, int D) {
  const int top = cy - D, bottom = cy + D, left = cx - D, right = cx + D;
  const int bTop = top >= t->top, bBottom = bottom <= t->bottom, bLeft = left >= t->left, bRight = right <= t->right;
  t->round++;
  if (D == 1) {
    if (bTop) probe(t, cx, top, 2, 1);
    if (bLeft) probe(t, left, cy, 4, 1);
    if (bRight) probe(t, right, cy, 5, 1);
    if (bBottom) probe(t, cx, bottom, 7, 1);
  } else if (D <= 8) {
    const int h = D >> 1, top2 = cy - h, bottom2 = cy + h, left2 = cx - h, right2 = cx + h;
    if (bTop && bBottom && bLeft && bRight) {
      probe(t, cx, top, 2, D);
      probe(t, left2, top2, 1, h);
      probe(t, right2, top2, 3, h);
      probe(t, left, cy, 4, D);
      probe(t, right, cy, 5, D);
      probe(t, left2, bottom2, 6, h);
      probe(t, right2, bottom2, 8, h);
      probe(t, cx, bottom, 7, D);
    } else {
      if (bTop) probe(t, cx, top, 2, D);
      if (top2 >= t->top) {
        if (left2 >= t->left) probe(t, left2, top2, 1, h);
        if (right2 <= t->right) probe(t, right2, top2, 3, h);
      }
      if (bLeft) probe(t, left, cy, 4, D);
      if (bRight) probe(t, right, cy, 5, D);
      if (bottom2 <= t->bottom) {
        if (left2 >= t->left) probe(t, left2, bottom2, 6, h);
        if (right2 <= t->right) probe(t, right2, bottom2, 8, h);
      }
      if (bBottom) probe(t, cx, bottom, 7, D);
    }
  } else {
    int k;
    if (bTop && bBottom && bLeft && bRight) {
      probe(t, cx, top, 0, D);
      probe(t, left, cy, 0, D);
      probe(t, right, cy, 0, D);
      probe(t, cx, bottom, 0, D);
      for (k = 1; k < 4; k++) {
        const int yt = top + (D >> 2) * k, yb = bottom - (D >> 2) * k, xl = cx - (D >> 2) * k, xr = cx + (D >> 2) * k;
        probe(t, xl, yt, 0, D);
        probe(t, xr, yt, 0, D);
        probe(t, xl, yb, 0, D);
        probe(t, xr, yb, 0, D);
      }
    } else {
      if (bTop) probe(t, cx, top, 0, D);
      if (bLeft) probe(t, left, cy, 0, D);
      if (bRight) probe(t, right, cy, 0, D);
      if (bBottom) probe(t, cx, bottom, 0, D);
      for (k = 1; k < 4; k++) {
        const int yt = top + (D >> 2) * k, yb = bottom - (D >> 2) * k, xl = cx - (D >> 2) * k, xr = cx + (D >> 2) * k;
        if (yt >= t->top) {
          if (xl >= t->left) probe(t, xl, yt, 0, D);
          if (xr <= t->right) probe(t, xr, yt, 0, D);
        }
        if (yb <= t->bottom) {
          if (xl >= t->left) probe(t, xl, yb, 0, D);
          if (xr <= t->right) probe(t, xr, yb, 0, D);
        }
      }
    }
  }
}

/* xTZ2PointSearch */
static void two_point(Tz* t) {
  const int cx = t->bx, cy = t->by;
  const int L = cx - 1 >= t->left, R = cx + 1 <= t->right, T = cy - 1 >= t->top, B = cy + 1 <= t->bottom;
  switch (t->pt) {
    case 1: if (L) probe(t, cx - 1, cy, 0, 2); if (T) probe(t, cx, cy - 1, 0, 2); break;
    case 2: if (T) { if (L) probe(t, cx - 1, cy - 1, 0, 2); if (R) probe(t, cx + 1, cy - 1, 0, 2); } break;
    case 3: if (T) probe(t, cx, cy - 1, 0, 2); if (R) probe(t, cx + 1, cy, 0, 2); break;
    case 4: if (L) { if (B) probe(t, cx - 1, cy + 1, 0, 2); if (T) probe(t, cx - 1, cy - 1, 0, 2); } break;
    case 5: if (R) { if (T) probe(t, cx + 1, cy - 1, 0, 2); if (B) probe(t, cx + 1, cy + 1, 0, 2); } break;
    case 6: if (L) probe(t, cx - 1, cy, 0, 2); if (B) probe(t, cx, cy + 1, 0, 2); break;
    case 7: if (B) { if (L) probe(t, cx - 1, cy + 1, 0, 2); if (R) probe(t, cx + 1, cy + 1, 0, 2); } break;
    case 8: if (R) probe(t, cx + 1, cy, 0, 2); if (B) probe(t, cx, cy + 1, 0, 2); break;
    default: break;
  }
}

static int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }

/* One PU.  desc[21]: the cucd_tz_desc fields (x, y, w, h, ref_idx, left, right, top, bottom, sub_shift, pred_x, pred_y, lambda, flags,
 * search_range, clip_left, clip_right, clip_top, clip_bottom, mv2n_x, mv2n_y); x, y, ref_idx are not read: refAtZeroMv is the PU's
 * co-located reference sample.  SADs: oracle_sad_surface on 1x1 windows, or (surf != NULL) surf[(y - sTop) * (sRight - sLeft + 1) +
 * x - sLeft], which must cover every probe.  The generic widths' SAD ignores sub_shift, as cucd_me_sad_surface does.
 * res[6] = mvx, mvy, sad, qmvx, qmvy, frac_cost (cucd_search_result).  trace (may be NULL): probe k is (x, y, p, d, stage, c) at
 * trace[6 k], for k < traceCap; stage 0 start points, 1 first search, 2 its two-point search, 3 raster, 4 + 2 i the diamonds of star
 * iteration i, 5 + 2 i its two-point search.  *nProbes (may be NULL) = number of probes.
 * Returns 0; -2 when the surface misses a probe; -3 when FRAC is asked without org / ref. */
int oracle_me_tz_search(int bitDepth, const int16_t* org, int orgStride, const int16_t* refAtZeroMv, int refStride, const int32_t* desc, const uint32_t* surf,
                        int sLeft, int sRight, int sTop, int sBottom, int32_t* res, int32_t* trace, int traceCap, int* nProbes) {
  Tz t;
  const int w = desc[2], h = desc[3], flags = desc[13], range = desc[14];
  const int cl = desc[15], cr = desc[16], ct = desc[17], cb = desc[18];
  int rl, rr, rt, rb, D, x, y, star = 0;
  t.bitDepth = bitDepth; t.org = org; t.orgStride = orgStride; t.w = w; t.h = h; t.ref = refAtZeroMv; t.refStride = refStride;
  t.subShift = (w == 4 || w == 8 || w == 12 || w == 16 || w == 24 || w == 32 || w == 48 || w == 64) ? desc[9] : 0;
  t.surf = surf; t.sl = sLeft; t.sr = sRight; t.st = sTop; t.sb = sBottom;
  t.lambda = (uint32_t)desc[12]; t.predX = desc[10]; t.predY = desc[11];
  t.left = desc[5]; t.right = desc[6]; t.top = desc[7]; t.bottom = desc[8];
  t.bx = t.by = 0; t.dist = t.round = t.pt = 0; t.best = 0xffffffffu;
  t.trace = trace; t.cap = traceCap; t.n = 0; t.stage = 0; t.err = 0;

  /* start points */
  probe(&t, clampi(t.predX, 4 * cl, 4 * cr) >> 2, clampi(t.predY, 4 * ct, 4 * cb) >> 2, 0, 0);
  probe(&t, 0, 0, 0, 0);
  rl = t.left; rr = t.right; rt = t.top; rb = t.bottom;
  if (flags & 4) {
    probe(&t, clampi(desc[19], cl, cr), clampi(desc[20], ct, cb), 0, 0);
    rl = clampi(t.bx - range, cl, cr); rr = clampi(t.bx + range, cl, cr); rt = clampi(t.by - range, ct, cb); rb = clampi(t.by + range, ct, cb);
  }
  /* first search */
  {
    const int cx = t.bx, cy = t.by;
    t.stage = 1;
    for (D = 1; D <= range; D *= 2) {
      diamond(&t, cx, cy, D);
      if (t.round >= 3) break;
    }
  }
  if (t.dist == 1) { t.dist = 0; t.stage = 2; two_point(&t); }
  /* raster */
  if (t.dist > 5) {
    t.dist = 5; t.stage = 3;
    for (y = rt; y <= rb; y += 5)
      for (x = rl; x <= rr; x += 5) probe(&t, x, y, 0, 5);
  }
  /* star refinement */
  while (t.dist > 0) {
    const int cx = t.bx, cy = t.by;
    t.dist = 0; t.pt = 0; t.stage = 4 + 2 * star;
    for (D = 1; D <= range; D *= 2) diamond(&t, cx, cy, D);
    if (t.dist == 1) { t.dist = 0; t.stage = 5 + 2 * star; if (t.pt != 0) two_point(&t); }
    star++;
  }
  if (t.err) return -2;
  if (nProbes) *nProbes = t.n;
  res[0] = t.bx; res[1] = t.by; res[2] = (int32_t)(t.best - oracle_mv_cost(t.lambda, t.bx, t.by, 2, t.predX, t.predY));
  res[3] = 4 * t.bx; res[4] = 4 * t.by; res[5] = 0;
  if (flags & 1) {
    uint32_t T[49], fc;
    int32_t qmv[2];
    if (!org || !refAtZeroMv) return -3;
    oracle_subpel_surface(bitDepth, org, orgStride, w, h, refAtZeroMv, refStride, t.bx, t.by, (flags & 2) ? 1 : 0, T);
    oracle_me_frac_walk(T, t.bx, t.by, t.predX, t.predY, t.lambda, qmv, &fc);
    res[3] = qmv[0]; res[4] = qmv[1]; res[5] = (int32_t)fc;
  }
  return 0;
}
