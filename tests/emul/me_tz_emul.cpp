// me_tz_emul.cpp - CPU replay of me_tz_kernel (csrc/me_kernels.cu) for one job (TEST HARNESS, not a product path).
//
// The kernel is one warp per job around the host/device phases of csrc/me_core.cuh: me_tz_walk drives the stages, and the warp
// evaluates a stage in chunks of 32 / G points (G = me_tz_lanes lanes per probe, me_tz_sad_part each), sums a group's parts with an
// xor butterfly inside the group, then reduces every segment of the chunk with an xor butterfly across the groups and folds each
// completed segment with me_tz_fold.  This file runs the same code for the 32 lane ids of one warp, with the two butterflies written
// out over arrays, and records every point of every folded segment (the points the walk's state depends on).
#include <cstdint>
#include <cstring>
#include <vector>
#include "me_core.cuh"

using namespace cucd;

extern "C" {

// desc[21]: the cucd_tz_desc fields; cur: the PU's source block (stride curStride); ref: the co-located sample (mv 0) of the padded
// reference plane.  res[6]: the integer result (qmv = 4 mv, frac_cost 0: the refinement is cucd_me_search's, replayed elsewhere).
// trace[6 k] = (x, y, p, d, stage, c) of the k-th point of the folded segments (stage numbers of tests/me_tz_oracle.c), at most cap.
// Returns the number of trace entries (-1 when the lanes of a warp disagree on a segment's key); *evaluated = every point the chunks evaluated (folded or not), *lanes = G.
int emul_me_tz_search(int bitDepth, const int16_t* cur, int curStride, const int16_t* ref, int refStride, const int32_t* desc, int32_t* res, int32_t* trace, int cap,
                      int* evaluated, int* lanes) {
  MeTzJob j{};
  j.w = (int16_t)desc[2]; j.h = (int16_t)desc[3];
  j.subShift = (int16_t)(me_width_is_hm(desc[2]) ? desc[9] : 0); j.flags = (int16_t)desc[13];
  j.left = (int16_t)desc[5]; j.right = (int16_t)desc[6]; j.top = (int16_t)desc[7]; j.bottom = (int16_t)desc[8];
  j.range = (int16_t)desc[14]; j.clipL = (int16_t)desc[15]; j.clipR = (int16_t)desc[16]; j.clipT = (int16_t)desc[17]; j.clipB = (int16_t)desc[18];
  j.mv2nX = (int16_t)desc[19]; j.mv2nY = (int16_t)desc[20];
  const MeSearchCost c{(uint32_t)desc[12], desc[10], desc[11], -1};
  const int w = j.w, nr = (j.h + (1 << j.subShift) - 1) >> j.subShift;
  std::vector<int16_t> sCur((size_t)nr * w);
  for (int lane = 0; lane < 32; lane++)                                 // the warp's staging loop
    for (int s = lane; s < nr * w; s += 32) { const int r = s / w; sCur[s] = cur[(size_t)(r << j.subShift) * curStride + s - r * w]; }
  const int G = me_tz_lanes(nr * w), P = 32 / G;
  int n = 0, stageNo = 0, star = -1;
  bool bad = false;
  *evaluated = 0; *lanes = G;
  const MeTzState st = me_tz_walk(j, c, [&](const MeTzStage& s, MeTzState& state) {
    if (s.kind == kTzStart) stageNo = 0;
    else if (s.kind == kTzDiamonds) stageNo = s.stop ? 1 : 4 + 2 * ++star;
    else if (s.kind == kTzTwo) stageNo = star < 0 ? 2 : 5 + 2 * star;
    else stageNo = 3;
    unsigned long long pend = kMeNoKey;
    std::vector<uint32_t> value(s.n > 0 ? s.n : 1);                     // c of every evaluated point, for the trace
    for (int base = 0; base < s.n; base += P) {
      const int end = base + P < s.n ? base + P : s.n;
      uint32_t part[32];
      unsigned long long key[32];
      MeTzPoint q[32];
      for (int lane = 0; lane < 32; lane++) {
        const int i = base + lane / G;
        q[lane].ok = false;
        if (i < s.n) q[lane] = me_tz_point(s, i);
        part[lane] = q[lane].ok ? me_tz_sad_part(sCur.data(), ref + (long long)q[lane].y * refStride + q[lane].x, refStride, w, nr, j.subShift, lane & (G - 1), G) : 0u;
      }
      for (int m = 1; m < G; m <<= 1) {                                // xor butterfly inside the groups
        uint32_t nx[32];
        for (int l = 0; l < 32; l++) nx[l] = part[l] + part[l ^ m];
        std::memcpy(part, nx, sizeof(nx));
      }
      for (int lane = 0; lane < 32; lane++) {
        const int i = base + lane / G;
        key[lane] = q[lane].ok ? ((unsigned long long)me_tz_probe_cost(part[lane], j.subShift, bitDepth, c, q[lane].x, q[lane].y) << 32) | (uint32_t)i : kMeNoKey;
        if (q[lane].ok && (lane & (G - 1)) == 0) { ++*evaluated; value[i] = (uint32_t)(key[lane] >> 32); }
      }
      const int k1 = me_tz_seg_of(s, end - 1);
      for (int k = me_tz_seg_of(s, base); k <= k1; k++) {
        unsigned long long kk[32];
        for (int lane = 0; lane < 32; lane++) { const int i = base + lane / G; kk[lane] = i < end && me_tz_seg_of(s, i) == k ? key[lane] : kMeNoKey; }
        for (int m = G; m < 32; m <<= 1) {                             // xor butterfly across the groups
          unsigned long long nx[32];
          for (int l = 0; l < 32; l++) nx[l] = me_key_min(kk[l], kk[l ^ m]);
          std::memcpy(kk, nx, sizeof(nx));
        }
        for (int l = 1; l < 32; l++) bad = bad || kk[l] != kk[0];      // every lane holds the segment's key
        pend = me_key_min(pend, kk[0]);
        if (me_tz_seg_first(s, k + 1) <= end) {
          for (int i = me_tz_seg_first(s, k); i < me_tz_seg_first(s, k + 1); i++) {
            const MeTzPoint p = me_tz_point(s, i);
            if (!p.ok) continue;
            if (n < cap) {
              int32_t* e = trace + 6 * n;
              e[0] = p.x; e[1] = p.y; e[2] = p.p; e[3] = p.d; e[4] = stageNo;
              e[5] = (int32_t)value[i];
            }
            n++;
          }
          const bool stop = me_tz_fold(state, s, pend);
          pend = kMeNoKey;
          if (stop) return;
        }
      }
    }
  });
  res[0] = st.bx; res[1] = st.by; res[2] = (int32_t)(st.best - me_mv_cost(c, st.bx, st.by, 2)); res[3] = 4 * st.bx; res[4] = 4 * st.by; res[5] = 0;
  return bad ? -1 : n;
}

}  // extern "C"
