// me_kernels.cu - integer-pel motion-estimation SAD surfaces on sm_100a.
//
// Replaces the distortion part of TEncSearch::xTZSearchHelp (TEncSearch.cpp:336-437) and of the
// full/raster search xPatternSearch (:3886-3943): for a PU and an inclusive integer MV window the
// kernel returns SAD(cur PU, ref + mv) for EVERY mv, computed exactly like TComRdCost::xGetSAD*
// (TComRdCost.cpp:465-962): rows stepped by 1<<subShift, sum << subShift, then >> (bitDepth-8).
// The host walks the TZ pattern over the table and adds getCost(mv) itself, so ties break as in HM.
//
// A surface is cut into tiles (me_core.cuh, me_enum_tiles).  The bulk of a window of 32 x 32 candidates or more goes to
// me_sad_dy_kernel (tiles M / E, "dy lanes": a thread owns eight candidates that slide over the same staged reference words);
// small windows, the last rows % 32 rows and caller-supplied (signed) source blocks go to the dx-lane kernels below (tiles O):
// one CTA = one 32x8 (32x16 for bytes) tile of candidates of one PU, the PU and the reference window staged once in shared memory,
// a lane owns one dx, a warp one dy.  9/10-bit content: samples as packed int16 pairs, |a-b| per half = max-min (VIMNMX.S16x2 x2 +
// ISUB), accumulated with IDP.2A.  8-bit content (me_sad_u8_kernel): samples as bytes, VABSDIFF4.U8.ACC.
#include <cuda_runtime.h>
#include "me_core.cuh"
#include "kernels.h"

namespace cucd {

constexpr int kMeTileX = 32, kMeTileY = 8;
constexpr int kMeRefPitch = 64 + kMeTileX + 4;       // int16 per staged reference row (even)
constexpr int kMeRefRows = 64 + kMeTileY;

// SIGNED: the source blocks are caller-supplied and may hold any int16 (the bi-predictive search compares 2 * org - other prediction,
// TEncSearch.cpp:3787-3797): |a - b| per half through the signed SIMD intrinsic instead of max - min of packed words, whose 32-bit
// subtraction would borrow across the halves for negative samples.  A half of that difference reaches 65535 (key -32768 against a
// reference sample of 32767), so the halves are summed as unsigned (IDP.2A.U16): the signed form would read 32768 .. 65535 as negative.
// OUT (all three SAD kernels): Surface stores every candidate's SAD at out[outOff + dy * cols + dx]; Argmin folds the candidates
// of a warp into the least search key (me_core.cuh, me_search_key) and commits it to am.keys[job] instead.
template <bool SIGNED, MeOut OUT = MeOut::Surface>
__global__ void __launch_bounds__(256)
me_sad_kernel(const MePlanes mp, const MeJob* __restrict__ jobs, const int32_t* __restrict__ tileJob, const int32_t* __restrict__ tileIdx,
              uint32_t* __restrict__ out, const MeArgmin am) {
  __shared__ __align__(16) int16_t sCur[64 * 64];
  __shared__ __align__(16) int16_t sRef[kMeRefRows * kMeRefPitch];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const MeJob job = jobs[tileJob[blockIdx.x]];
  const int cols = job.right - job.left + 1, rows = job.bottom - job.top + 1;
  int kind, dx0, dy0;                                                          // tile origin relative to (left, top)
  me_tile_unpack(tileIdx[blockIdx.x], kind, dx0, dy0);
  (void)kind;
  const int w = job.w, h = job.h;

  const int16_t* cur = mp.cur + job.curOff;
  const int curStride = mp.curStride ? mp.curStride : w;               // 0: caller-supplied blocks, w x h each, back to back
  for (int i = tid; i < w * h; i += 256) { const int y = i / w, x = i - y * w; sCur[y * w + x] = cur[(size_t)y * curStride + x]; }
  const int refStride = mp.refStride[job.refSlot];
  const int16_t* ref = mp.ref[job.refSlot] + job.refOff + (long long)(job.top + dy0) * refStride + (job.left + dx0);
  const int winW = min(w + kMeTileX - 1, w + cols - dx0 - 1), winH = min(h + kMeTileY - 1, h + rows - dy0 - 1);
  for (int i = tid; i < kMeRefRows * kMeRefPitch; i += 256) {
    const int y = i / kMeRefPitch, x = i - y * kMeRefPitch;
    sRef[i] = (y < winH && x < winW) ? ref[(long long)y * refStride + x] : (int16_t)0;
  }
  __syncthreads();

  const int dx = dx0 + lane, dy = dy0 + warp;
  if (OUT == MeOut::Surface && (dx >= cols || dy >= rows)) return;   // Argmin: every lane joins the warp's key reduction
  const int step = 1 << job.subShift;
  const uint32_t* cw = reinterpret_cast<const uint32_t*>(sCur);
  const uint32_t* rw = reinterpret_cast<const uint32_t*>(sRef);
  const uint32_t e16 = ((uint32_t)lane & 1u) << 4;
  const int pairs = w >> 1;
  int acc = 0;
  for (int y = 0; y < h; y += step) {
    const int rbase = ((y + warp) * kMeRefPitch + lane) >> 1;
    const int cbase = (y * w) >> 1;
    uint32_t prev = rw[rbase];
    for (int j = 0; j < pairs; j++) {
      const uint32_t next = rw[rbase + j + 1];
      const uint32_t r = funnel_r(prev, next, e16);
      const uint32_t c = cw[cbase + j];
      if constexpr (SIGNED) acc = (int)__dp2a_lo(__vabsdiffs2(c, r), 0x0101u, (uint32_t)acc);
      else acc = __dp2a_lo((int)(__vmaxs2(c, r) - __vmins2(c, r)), 0x0101, acc);
      prev = next;
    }
  }
  const uint32_t sad = ((uint32_t)acc << job.subShift) >> (mp.bitDepth - 8);
  if constexpr (OUT == MeOut::Surface) out[job.outOff + (long long)dy * cols + dx] = sad;
  else {
    const int ji = tileJob[blockIdx.x];
    me_key_warp_commit(dx < cols && dy < rows ? me_search_key(sad, dx, dy, cols, job.left, job.top, am.cost[ji]) : kMeNoKey, lane, am.keys + ji);
  }
}

// 8-bit content: the same tile of candidates with samples staged as BYTES - four absolute differences and their accumulation are one
// VABSDIFF4.U8.ACC, the unaligned reference word of a candidate is two aligned shared-memory words + one PRMT (the second word is
// the next iteration's first), the source word is a broadcast load: ~1.1 instructions per sample instead of 3.5.
constexpr int kMe8Pitch = 64 + kMeTileX + 8;         // bytes per staged reference row (multiple of 4, >= w + 31 + 4)
constexpr int kMe8TileY = 16;                        // candidate rows per CTA: a thread owns dy = warp and warp + 8 (they share the source loads)
constexpr int kMe8RefRows = 64 + kMe8TileY;

template <MeOut OUT = MeOut::Surface>
__global__ void __launch_bounds__(256)
me_sad_u8_kernel(const MePlanes mp, const MeJob* __restrict__ jobs, const int32_t* __restrict__ tileJob, const int32_t* __restrict__ tileIdx,
                 uint32_t* __restrict__ out, const MeArgmin am) {
  __shared__ __align__(16) uint8_t sCur[64 * 64];
  __shared__ __align__(16) uint8_t sRef[kMe8RefRows * kMe8Pitch];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const MeJob job = jobs[tileJob[blockIdx.x]];
  const int cols = job.right - job.left + 1, rows = job.bottom - job.top + 1;
  int kind, dx0, dy0;
  me_tile_unpack(tileIdx[blockIdx.x], kind, dx0, dy0);
  (void)kind;
  const int w = job.w, h = job.h;
  const int step = 1 << job.subShift;

  // staging: a warp per row, lanes along the row (no divisions); only the rows the sub-sampled SAD reads
  const int16_t* cur = mp.cur + job.curOff;
  for (int y = warp * step; y < h; y += 8 * step)
    for (int x = lane; x < w; x += 32) sCur[y * w + x] = (uint8_t)cur[(size_t)y * mp.curStride + x];
  const int refStride = mp.refStride[job.refSlot];
  const int16_t* ref = mp.ref[job.refSlot] + job.refOff + (long long)(job.top + dy0) * refStride + (job.left + dx0);
  const int winW = min(w + kMeTileX - 1, w + cols - dx0 - 1), winH = min(h + kMe8TileY - 1, h + rows - dy0 - 1);
  for (int y = warp; y < winH; y += 8)
    for (int x = lane; x < winW; x += 32) sRef[y * kMe8Pitch + x] = (uint8_t)ref[(long long)y * refStride + x];
  __syncthreads();

  const int dx = dx0 + lane, dyA = dy0 + warp, dyB = dyA + 8;
  if (OUT == MeOut::Surface && (dx >= cols || dyA >= rows)) return;
  const bool hasB = dyB < rows;
  const uint32_t* cw = reinterpret_cast<const uint32_t*>(sCur);
  const uint32_t* rw = reinterpret_cast<const uint32_t*>(sRef);
  const uint32_t sel = 0x3210u + 0x1111u * ((uint32_t)lane & 3u);      // bytes (lane & 3) .. +3 of the 8-byte pair {lo, hi}
  const int words = w >> 2;                                            // w is a multiple of 4
  uint32_t accA = 0, accB = 0;
  for (int y = 0; y < h; y += step) {
    const int ra = ((y + warp) * kMe8Pitch + lane) >> 2;               // kMe8Pitch is a multiple of 4
    const int rb = hasB ? ra + 8 * (kMe8Pitch >> 2) : ra;              // rows beyond the window are not staged: keep the reads inside
    const int cbase = (y * w) >> 2;
    uint32_t pa = rw[ra], pb = rw[rb];
    for (int j = 0; j < words; j++) {
      const uint32_t c = cw[cbase + j];                                // broadcast
      const uint32_t na = rw[ra + j + 1], nb = rw[rb + j + 1];
      accA = me_sad4(c, __byte_perm(pa, na, sel), accA);
      accB = me_sad4(c, __byte_perm(pb, nb, sel), accB);
      pa = na; pb = nb;
    }
  }
  if constexpr (OUT == MeOut::Surface) {
    out[job.outOff + (long long)dyA * cols + dx] = accA << job.subShift;               // bitDepth 8: no final shift
    if (hasB) out[job.outOff + (long long)dyB * cols + dx] = accB << job.subShift;
  } else {
    const int ji = tileJob[blockIdx.x];
    const MeSearchCost& c = am.cost[ji];
    const bool okA = dx < cols && dyA < rows, okB = okA && hasB;
    const unsigned long long kA = okA ? me_search_key(accA << job.subShift, dx, dyA, cols, job.left, job.top, c) : kMeNoKey;
    me_key_warp_commit(me_key_min(kA, okB ? me_search_key(accB << job.subShift, dx, dyB, cols, job.left, job.top, c) : kMeNoKey), lane, am.keys + ji);
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Tiles M and E (me_core.cuh): lanes along dy.  All lanes of a warp share dx, hence the byte / half-word alignment of their
// reference words: an aligned word is one conflict-free shared-memory load (row pitch odd) + one PRMT / SHF, and it serves the eight
// candidates dx, dx + 4, ... (dx + 2, ... for 16-bit samples) of the thread as they slide along the row.  Per four 8-bit samples and
// candidate: 1 VABSDIFF4.U8.ACC + 3/8 of a load / permute instead of 3.5 instructions; per two 16-bit samples: VIMNMX.S16x2 + two
// packed additions (sum c + sum r - 2 sum min) instead of 7.  Results leave through shared memory as 128-byte rows of the surface.
// ---------------------------------------------------------------------------------------------------------------------
template <bool U8, MeOut OUT = MeOut::Surface>
__global__ void __launch_bounds__(256)
me_sad_dy_kernel(const MePlanes mp, const MeJob* __restrict__ jobs, const int32_t* __restrict__ tileJob, const int32_t* __restrict__ tileIdx,
                 uint32_t* __restrict__ out, const MeArgmin am) {
  constexpr int P = U8 ? kMeDyPitch8 : kMeDyPitch16, SPW = U8 ? 4 : 2;
  __shared__ __align__(16) uint32_t sCur[64 * 64 / SPW];
  __shared__ __align__(16) uint32_t sRef[kMeDyRows * P];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const MeJob job = jobs[tileJob[blockIdx.x]];
  const int cols = job.right - job.left + 1, rows = job.bottom - job.top + 1;
  int kind, x0, y0;
  me_tile_unpack(tileIdx[blockIdx.x], kind, x0, y0);
  const int w = job.w, h = job.h, step = 1 << job.subShift;
  const MeDyTile tl = me_dy_tile(kind, x0, y0, w, h, cols, rows);

  me_dy_stage_cur<U8>(warp, lane, mp.cur + job.curOff, mp.curStride, w, h, step, sCur);
  const int refStride = mp.refStride[job.refSlot];
  me_dy_stage_ref<U8>(warp, lane, mp.ref[job.refSlot] + job.refOff + (long long)(job.top + y0) * refStride + (job.left + x0), refStride, tl.winW, tl.winH, sRef);
  __syncthreads();

  const MeDyWarp q = me_dy_warp<U8>(kind, warp, tl.cr);
  const int lam = 32 * q.blk + lane;
  const bool work = q.active && 32 * q.blk < tl.nLam;                  // warp uniform
  const int shiftOut = U8 ? 0 : mp.bitDepth - 8;
  if (kind == kMeKindM) {
    uint32_t sad[kMeDyK];
    if (work) {
      if (U8) me_dy_sad_u8<kMeDyK>(sCur, sRef, w >> 2, h, step, lam, q.wbase, q.s, sad);
      else me_dy_sad_s16<kMeDyK>(sCur, sRef, w >> 1, h, step, lam, q.wbase, q.s, me_fold_rows(mp.bitDepth, w >> 1), sad);
    }
    if constexpr (OUT == MeOut::Argmin) {                              // `work` is warp uniform
      // the tile origin is read again here, not kept live across the SAD runs (no spill at 64 registers)
      int k2, xr, yr;
      me_tile_unpack(*(const volatile int32_t*)&tileIdx[blockIdx.x], k2, xr, yr);
      if (work) me_key_warp_commit(me_dy_lane_key<kMeDyK, SPW>(sad, job.subShift, shiftOut, lam < tl.nLam, xr + q.delta0, yr + lam, cols, job.left, job.top,
                                                              am.cost[tileJob[blockIdx.x]]), lane, am.keys + tileJob[blockIdx.x]);
      return;
    }
    __syncthreads();                                                   // the staged window is dead: its space carries the tile out
    if (work) {
#pragma unroll
      for (int k = 0; k < kMeDyK; k++) sRef[lam * 33 + q.delta0 + SPW * k] = (sad[k] << job.subShift) >> shiftOut;
    }
    __syncthreads();
    for (int i = tid; i < tl.nLam * 32; i += 256) {
      const int r = i >> 5, c = i & 31;
      out[job.outOff + (long long)(y0 + r) * cols + x0 + c] = sRef[r * 33 + c];
    }
  } else {
    if (!work) return;
    uint32_t sad[1];
    if (U8) me_dy_sad_u8<1>(sCur, sRef, w >> 2, h, step, lam, q.wbase, q.s, sad);
    else me_dy_sad_s16<1>(sCur, sRef, w >> 1, h, step, lam, q.wbase, q.s, me_fold_rows(mp.bitDepth, w >> 1), sad);
    if constexpr (OUT == MeOut::Argmin) {
      int k2, xr, yr;
      me_tile_unpack(*(const volatile int32_t*)&tileIdx[blockIdx.x], k2, xr, yr);
      me_key_warp_commit(me_dy_lane_key<1, SPW>(sad, job.subShift, shiftOut, lam < tl.nLam, xr + q.delta0, yr + lam, cols, job.left, job.top, am.cost[tileJob[blockIdx.x]]),
                         lane, am.keys + tileJob[blockIdx.x]);
    } else if (lam < tl.nLam) out[job.outOff + (long long)(y0 + lam) * cols + x0 + q.delta0] = (sad[0] << job.subShift) >> shiftOut;
  }
}

// ---------------------------------------------------------------------------------------------------------------------
// Fractional-pel refinement (SURVEY.md 8f.3): xPatternSearchFracDIF TEncSearch.cpp:4340-4376 = xExtDIFUpSamplingH / Q
// (:5431-5637) + xPatternRefinement (:808-865).  Every candidate block of the reference's half- and quarter-pel stages is the
// separable 8-tap luma interpolation (TComInterpolationFilter.cpp:57-290: rows into 14-bit intermediates, then columns with
// rounding and clipping; filterCopy for zero fractions) of the reference at that quarter-pel position, compared with the source
// block by xGetHADs (8x8 tiles when both sizes are multiples of 8, else 4x4) or xGetSAD.  The kernel returns the distortion of all
// 49 positions within +-3 quarter pels of the integer MV; the host walks the two 9-point stages and adds getCost(mv).
// One CTA = one PU and one horizontal offset dx: the reference window is staged once, filtered horizontally once, and the seven
// vertical offsets reuse those intermediates.
// ---------------------------------------------------------------------------------------------------------------------
__constant__ int8_t kLumaFilter[4][8] = {{0, 0, 0, 64, 0, 0, 0, 0}, {-1, 4, -10, 58, 17, -5, 1, 0}, {-1, 4, -11, 40, 40, -11, 4, -1}, {0, 1, -5, 17, 58, -10, 4, -1}};

// T x T Hadamard cost of (a - b) tiles with T lanes per tile (one tile row each): rows transformed in registers, columns across the
// lanes with shuffles; every lane of the warp takes part (tasks past the end carry zeros).  Returns the tile's HM-rounded cost in the
// tile's first lane, 0 elsewhere.  Only sum |coefficient| matters (TComRdCost.cpp:1343-1534), so butterfly order and signs are free.
template <int T>
__device__ __forceinline__ int hadamard_tile_rows(const int16_t* a, const int16_t* b, int pitch, int tile, int tilesX, bool valid, int lane) {
  const int r = lane & (T - 1);
  int v[T];
  if (valid) {
    const int o = ((tile / tilesX) * T + r) * pitch + (tile % tilesX) * T;
#pragma unroll
    for (int x = 0; x < T; x++) v[x] = a[o + x] - b[o + x];
  } else {
#pragma unroll
    for (int x = 0; x < T; x++) v[x] = 0;
  }
#pragma unroll
  for (int len = 1; len < T; len <<= 1)
#pragma unroll
    for (int j = 0; j < T; j++)
      if (!(j & len)) { const int p = v[j], q = v[j + len]; v[j] = p + q; v[j + len] = p - q; }
#pragma unroll
  for (int m = 1; m < T; m <<= 1) {
    const bool upper = (r & m) != 0;
#pragma unroll
    for (int x = 0; x < T; x++) { const int other = __shfl_xor_sync(0xffffffffu, v[x], m); v[x] = upper ? other - v[x] : v[x] + other; }
  }
  int s = 0;
#pragma unroll
  for (int x = 0; x < T; x++) s += abs(v[x]);
#pragma unroll
  for (int m = 1; m < T; m <<= 1) s += __shfl_xor_sync(0xffffffffu, s, m);
  if (r != 0) return 0;
  return T == 8 ? (s + 2) >> 2 : (s + 1) >> 1;               // xCalcHADs8x8 / xCalcHADs4x4 rounding
}

constexpr int kSpWinPitch = 64 + 10;      // int16 per staged window row (w + 9 <= 73)

__global__ void __launch_bounds__(256)
me_subpel_kernel(const MePlanes mp, const SubpelJob* __restrict__ jobs, uint32_t* __restrict__ out) {
  __shared__ __align__(16) int16_t sCur[64 * 64];
  __shared__ __align__(16) int16_t sWin[(64 + 9) * kSpWinPitch];
  __shared__ __align__(16) int16_t sHor[(64 + 9) * 64];
  __shared__ __align__(16) int16_t sPred[64 * 64];
  __shared__ int sSum[8];
  const int tid = threadIdx.x;
  const SubpelJob job = jobs[blockIdx.x];
  const int w = job.w, h = job.h, bd = mp.bitDepth, head = 14 - bd;
  if (mp.curStride != 0 && subpel_is_small(w, h)) return;            // me_subpel_small_kernel's PU (block uniform)
  const int dx = (int)blockIdx.y - 3, ix = dx >> 2, fx = dx & 3;

  const int16_t* cur = mp.cur + job.curOff;
  const int curStride = mp.curStride ? mp.curStride : w;               // 0: caller-supplied blocks (bi-predictive refinement)
  // i / w and i / (w + 9) as one IMAD.HI: exact for i * d < 2^32 (i < 6000, d <= 73)
  const uint32_t invW = 0xffffffffu / (uint32_t)w + 1u, invW9 = 0xffffffffu / (uint32_t)(w + 9) + 1u;
  for (int i = tid; i < w * h; i += 256) { const int y = (int)__umulhi((uint32_t)i, invW), x = i - y * w; sCur[i] = cur[(size_t)y * curStride + x]; }
  const int refStride = mp.refStride[job.refSlot];
  const int16_t* ref = mp.ref[job.refSlot] + job.refOff - 4 * (long long)refStride - 4;       // window origin (-4, -4) from the integer MV position
  for (int i = tid; i < (h + 9) * (w + 9); i += 256) { const int y = (int)__umulhi((uint32_t)i, invW9), x = i - y * (w + 9); sWin[y * kSpWinPitch + x] = ref[(long long)y * refStride + x]; }
  __syncthreads();
  // rows of the window -> 14-bit intermediates at horizontal fraction fx (filterHor, isFirst, !isLast)
  for (int i = tid; i < (h + 9) * w; i += 256) {
    const int r = (int)__umulhi((uint32_t)i, invW), c = i - r * w;
    const int16_t* s = &sWin[r * kSpWinPitch + c + 4 + ix];
    int v;
    if (fx == 0) v = (s[0] << head) - 8192;
    else {
      int sum = 0;
#pragma unroll
      for (int k = 0; k < 8; k++) sum += s[k - 3] * kLumaFilter[fx][k];
      v = (sum - (8192 << (6 - head))) >> (6 - head);
    }
    sHor[r * w + c] = (int16_t)v;
  }
  __syncthreads();
  const bool tile8 = !(w & 7) && !(h & 7);
  const int T = tile8 ? 8 : 4, tilesX = w / T, nTiles = tilesX * (h / T);
  // Small PUs leave most of the CTA idle (an 8x8 PU is 64 samples, 8 Hadamard lanes): G vertical offsets share one pass of the
  // column filter / distortion / reduction, so that such a PU takes 2 passes (3 barriers each) instead of 7.
  const int wh = w * h;
  const int G = wh >= 256 ? 1 : (256 / wh < 7 ? 256 / wh : 7);
  for (int dyBase = -3; dyBase <= 3; dyBase += G) {
    const int nG = 4 - dyBase < G ? 4 - dyBase : G;
    if (tid < nG) sSum[tid] = 0;
    for (int i = tid; i < nG * wh; i += 256) {               // columns (filterVer, !isFirst, isLast)
      const int g = G == 1 ? 0 : i / wh, rem = i - g * wh;
      const int r = (int)__umulhi((uint32_t)rem, invW), c = rem - r * w;
      const int dy = dyBase + g, iy = dy >> 2, fy = dy & 3;
      const int16_t* s = &sHor[(r + 4 + iy) * w + c];
      int v;
      if (fy == 0) v = (s[0] + 8192 + (1 << (head - 1))) >> head;
      else {
        int sum = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) sum += s[(k - 3) * w] * kLumaFilter[fy][k];
        v = (sum + (1 << (5 + head)) + (8192 << 6)) >> (6 + head);
      }
      sPred[i] = (int16_t)min(max(v, 0), (1 << bd) - 1);
    }
    __syncthreads();
    if (G == 1) {
      int part = 0;
      if (job.useHadamard) {
        const int nTasks = nTiles * T;                        // T lanes per tile; whole warps iterate so that every lane joins the shuffles
        for (int base = (tid & ~31); base < nTasks; base += 256) {
          const int task = base + (tid & 31), tile = task / T;
          if (tile8) part += hadamard_tile_rows<8>(sCur, sPred, w, tile, tilesX, task < nTasks, tid & 31);
          else part += hadamard_tile_rows<4>(sCur, sPred, w, tile, tilesX, task < nTasks, tid & 31);
        }
      } else {
        for (int i = tid; i < wh; i += 256) part += abs(sCur[i] - sPred[i]);
      }
#pragma unroll
      for (int m = 16; m > 0; m >>= 1) part += __shfl_xor_sync(0xffffffffu, part, m);
      if ((tid & 31) == 0 && part) atomicAdd(&sSum[0], part);
    } else if (job.useHadamard) {                             // nG * nTiles * T <= 256 tasks: one pass, the tile's first lane adds to its offset's sum
      const int perG = nTiles * T, nTasks = nG * perG;
      if ((tid & ~31) < nTasks) {
        const int g = tid / perG, local = tid - g * perG, tile = local / T;
        const bool ok = tid < nTasks;
        const int16_t* pg = sPred + (ok ? g : 0) * wh;
        const int part = tile8 ? hadamard_tile_rows<8>(sCur, pg, w, tile, tilesX, ok, tid & 31) : hadamard_tile_rows<4>(sCur, pg, w, tile, tilesX, ok, tid & 31);
        if (ok && part) atomicAdd(&sSum[g], part);
      }
    } else {
      for (int i = tid; i < nG * wh; i += 256) { const int g = i / wh; const int d = abs(sCur[i - g * wh] - sPred[i]); if (d) atomicAdd(&sSum[g], d); }
    }
    __syncthreads();
    if (tid < nG) out[(size_t)blockIdx.x * 49 + (dyBase + tid + 3) * 7 + dx + 3] = (uint32_t)sSum[tid] >> (bd - 8);
    __syncthreads();
  }
}

// Small PUs (me_core.cuh, subpel_is_small): one CTA per PU, all 49 positions; the phases are the host/device functions the CPU replay runs.
__global__ void __launch_bounds__(256)
me_subpel_small_kernel(const MePlanes mp, const SubpelJob* __restrict__ jobs, uint32_t* __restrict__ out) {
  __shared__ __align__(16) int16_t sCur[256];
  __shared__ __align__(16) int16_t sWin[kSpSmallWinCap];
  __shared__ __align__(16) int16_t sHor[kSpHorCap];
  __shared__ __align__(16) int16_t sPred[kSpPredCap];
  __shared__ int sSum[64];
  const int tid = threadIdx.x;
  const SubpelJob job = jobs[blockIdx.x];
  if (!subpel_is_small(job.w, job.h)) return;                         // me_subpel_kernel's PU (block uniform)
  const SubpelGeo g = subpel_geo(job.w, job.h, mp.bitDepth);
  const int refStride = mp.refStride[job.refSlot];
  subpel_small_stage(tid, g, mp.cur + job.curOff, mp.curStride, mp.ref[job.refSlot] + job.refOff - 4 * (long long)refStride - 4, refStride, sCur, sWin);
  __syncthreads();
  subpel_small_hor(tid, g, sWin, sHor);
  __syncthreads();
  const int perGroup = kSpPredCap / g.wh < 49 ? kSpPredCap / g.wh : 49;
  for (int pBase = 0; pBase < 49; pBase += perGroup) {
    const int nP = 49 - pBase < perGroup ? 49 - pBase : perGroup;
    if (tid < nP) sSum[tid] = 0;
    subpel_small_ver(tid, g, pBase, nP, sHor, sPred);
    __syncthreads();
    subpel_small_dist(tid, g, nP, job.useHadamard, sCur, sPred, sSum);
    __syncthreads();
    if (tid < nP) out[(size_t)blockIdx.x * 49 + pBase + tid] = (uint32_t)sSum[tid] >> (mp.bitDepth - 8);
  }
}

// Motion compensation + distortion of inter candidates (me_core.cuh, me_mc_*): a CTA takes the candidates jobs[ctaFirst[b] ..
// ctaFirst[b + 1]) of one class; the predictions reuse the shared memory of the dead reference windows.
__global__ void __launch_bounds__(256)
me_mc_kernel(const MePlanes mp, const McJob* __restrict__ jobs, const int32_t* __restrict__ ctaFirst, uint32_t* __restrict__ dist, int16_t* __restrict__ pred) {
  __shared__ __align__(16) int16_t sCur[kMcCurCap];
  __shared__ __align__(16) int16_t sWin[kMcWinCap];
  __shared__ __align__(16) int16_t sTmp[kMcTmpCap];
  __shared__ int sSum[kMcMaxCand];
  const int tid = threadIdx.x;
  const int first = ctaFirst[blockIdx.x];
  const McJob* J = jobs + first;
  const McGeo g = me_mc_geo(J[0].w, J[0].h, J[0].nl, ctaFirst[blockIdx.x + 1] - first, mp.bitDepth);
  const int had = J[0].had;
  if (tid < g.n) sSum[tid] = 0;
  me_mc_stage(tid, g, J, mp.cur, mp.curStride, mp.ref, mp.refStride, sCur, sWin);
  __syncthreads();
  me_mc_hor(tid, g, J, sWin, sTmp);
  __syncthreads();
  me_mc_ver(tid, g, J, sTmp, sWin, pred);
  __syncthreads();
  subpel_small_dist(tid, subpel_geo(g.w, g.h, g.bd), g.n, had, sCur, sWin, sSum, g.wh);
  __syncthreads();
  if (tid < g.n) dist[J[tid].outIndex] = (uint32_t)sSum[tid] >> (g.bd - 8);
}

// 4:2:0 chroma motion compensation + SSE (me_core.cuh, me_mcc_*): a CTA takes the candidates jobs[ctaFirst[b] .. ctaFirst[b + 1]) of
// one class, both planes of each; the predictions reuse the shared memory of the dead reference windows.
__global__ void __launch_bounds__(256)
me_mc_chroma_kernel(const McChromaPlanes cp, const McJob* __restrict__ jobs, const int32_t* __restrict__ ctaFirst, uint32_t* __restrict__ sse,
                    int16_t* __restrict__ pred) {
  __shared__ __align__(16) int16_t sCur[kMcCurCap];
  __shared__ __align__(16) int16_t sWin[kMcWinCap];
  __shared__ __align__(16) int16_t sTmp[kMcTmpCap];
  __shared__ int sSum[2 * kMcMaxCand];
  const int tid = threadIdx.x;
  const int first = ctaFirst[blockIdx.x];
  const McJob* J = jobs + first;
  const McGeo g = me_mcc_geo(J[0].w, J[0].h, J[0].nl, ctaFirst[blockIdx.x + 1] - first, cp.bitDepth);
  if (tid < 2 * g.n) sSum[tid] = 0;
  me_mcc_stage(tid, g, J, cp.cur, cp.curStride, cp.ref, cp.refStride, sCur, sWin);
  __syncthreads();
  me_mcc_hor(tid, g, J, sWin, sTmp);
  __syncthreads();
  me_mcc_ver(tid, g, J, sTmp, sWin, pred);
  __syncthreads();
  me_mcc_sse(tid, g, sCur, sWin, sSum);
  __syncthreads();
  if (tid < 2 * g.n) sse[2 * J[tid >> 1].outIndex + (tid & 1)] = (uint32_t)sSum[tid];
}

cudaError_t launch_me_mc_chroma(const McChromaPlanes& cp, const McJob* jobs, const int32_t* ctaFirst, int nCta, uint32_t* sse, int16_t* pred, cudaStream_t st,
                                int* launches) {
  if (nCta <= 0) return cudaSuccess;
  me_mc_chroma_kernel<<<nCta, 256, 0, st>>>(cp, jobs, ctaFirst, sse, pred);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_me_mc(const MePlanes& mp, const McJob* jobs, const int32_t* ctaFirst, int nCta, uint32_t* dist, int16_t* pred, cudaStream_t st, int* launches) {
  if (nCta <= 0) return cudaSuccess;
  me_mc_kernel<<<nCta, 256, 0, st>>>(mp, jobs, ctaFirst, dist, pred);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

cudaError_t launch_me_subpel(const MePlanes& mp, const SubpelJob* jobs, int nJobs, uint32_t* out, cudaStream_t st, int* launches) {
  if (nJobs <= 0) return cudaSuccess;
  me_subpel_kernel<<<dim3(nJobs, 7), 256, 0, st>>>(mp, jobs, out);
  if (launches) *launches += 1;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || mp.curStride == 0) return e;                // caller-supplied key blocks: every PU stays with me_subpel_kernel
  me_subpel_small_kernel<<<nJobs, 256, 0, st>>>(mp, jobs, out);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// tile records: [0, nTilesDy) the dy-lane tiles (M, E), [nTilesDy, nTilesDy + nTilesO) the dx-lane tiles (O); the two launches write disjoint candidates
template <MeOut OUT>
static cudaError_t launch_sad_tiles(const MePlanes& mp, const MeJob* jobs, const int32_t* tileJob, const int32_t* tileIdx, int nTilesDy, int nTilesO, uint32_t* out,
                                    const MeArgmin& am, cudaStream_t st, int* launches) {
  if (nTilesDy > 0) {
    if (mp.curStride == 0) return cudaErrorInvalidValue;                // dy-lane tiles need the picture-resident (unsigned) source
    if (mp.bitDepth == 8) me_sad_dy_kernel<true, OUT><<<nTilesDy, 256, 0, st>>>(mp, jobs, tileJob, tileIdx, out, am);
    else me_sad_dy_kernel<false, OUT><<<nTilesDy, 256, 0, st>>>(mp, jobs, tileJob, tileIdx, out, am);
    if (launches) *launches += 1;
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  if (nTilesO <= 0) return cudaSuccess;
  tileJob += nTilesDy; tileIdx += nTilesDy;
  if (mp.curStride == 0) me_sad_kernel<true, OUT><<<nTilesO, 256, 0, st>>>(mp, jobs, tileJob, tileIdx, out, am);     // caller-supplied (possibly signed) source blocks
  else if (mp.bitDepth == 8) me_sad_u8_kernel<OUT><<<nTilesO, 256, 0, st>>>(mp, jobs, tileJob, tileIdx, out, am);
  else me_sad_kernel<false, OUT><<<nTilesO, 256, 0, st>>>(mp, jobs, tileJob, tileIdx, out, am);
  if (launches) *launches += 1;
  return cudaGetLastError();
}
cudaError_t launch_me_sad(const MePlanes& mp, const MeJob* jobs, int nJobs, const int32_t* tileJob, const int32_t* tileIdx, int nTilesDy, int nTilesO,
                          uint32_t* out, cudaStream_t st, int* launches) {
  (void)nJobs;
  return launch_sad_tiles<MeOut::Surface>(mp, jobs, tileJob, tileIdx, nTilesDy, nTilesO, out, MeArgmin{nullptr, nullptr}, st, launches);
}

// cucd_me_search: keys (~0, then the Argmin SAD kernels) -> prep -> sub-pel tables of the FRAC PUs -> walk
__global__ void __launch_bounds__(128)
me_search_prep_kernel(const MePlanes mp, const MeJob* __restrict__ jobs, int nJobs, const MeSearchCost* __restrict__ cost, const unsigned long long* __restrict__ keys,
                      const SubpelJob* __restrict__ subIn, SubpelJob* __restrict__ subOut, MeSearchOut* __restrict__ out) {
  const int i = blockIdx.x * 128 + threadIdx.x;
  if (i < nJobs) me_search_prep(i, keys, jobs, cost, mp.refStride, subIn, subOut, out);
}
__global__ void __launch_bounds__(128)
me_search_walk_kernel(const int32_t* __restrict__ fracJob, int nFrac, const MeSearchCost* __restrict__ cost, const uint32_t* __restrict__ tables,
                      MeSearchOut* __restrict__ out) {
  const int f = blockIdx.x * 128 + threadIdx.x;
  if (f >= nFrac) return;
  const int i = fracJob[f];
  MeSearchOut o = out[i];
  me_search_walk(tables + (size_t)f * 49, cost[i], o);
  out[i] = o;
}

cudaError_t launch_me_search(const MePlanes& mp, const MeJob* jobs, int nJobs, const int32_t* tileJob, const int32_t* tileIdx, int nTilesDy, int nTilesO,
                             const MeSearchCost* cost, unsigned long long* keys, const SubpelJob* subIn, SubpelJob* subDev, const int32_t* fracJob, int nFrac,
                             uint32_t* tables, MeSearchOut* out, cudaStream_t st, int* launches) {
  if (nJobs <= 0) return cudaSuccess;
  cudaError_t e = cudaMemsetAsync(keys, 0xff, (size_t)nJobs * sizeof(unsigned long long), st);
  if (e != cudaSuccess) return e;
  e = launch_sad_tiles<MeOut::Argmin>(mp, jobs, tileJob, tileIdx, nTilesDy, nTilesO, nullptr, MeArgmin{cost, keys}, st, launches);
  if (e != cudaSuccess) return e;
  me_search_prep_kernel<<<(nJobs + 127) / 128, 128, 0, st>>>(mp, jobs, nJobs, cost, keys, subIn, subDev, out);
  if (launches) *launches += 1;
  if ((e = cudaGetLastError()) != cudaSuccess || nFrac <= 0) return e;
  if ((e = launch_me_subpel(mp, subDev, nFrac, tables, st, launches)) != cudaSuccess) return e;
  me_search_walk_kernel<<<(nFrac + 127) / 128, 128, 0, st>>>(fracJob, nFrac, cost, tables, out);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

// cucd_me_tz_search (me_core.cuh, me_tz_*): warp `warp` of CTA b walks job ctaFirst[b] + warp.  Its source block (the rows the
// sub-sampled SAD reads) sits in shared memory, the reference samples come from the padded plane through the read-only path.
__global__ void __launch_bounds__(32 * kTzWarps)
me_tz_kernel(const MePlanes mp, const MeTzJob* __restrict__ jobs, const int32_t* __restrict__ ctaFirst, int maxSamples, const MeSearchCost* __restrict__ cost,
             const SubpelJob* __restrict__ subIn, SubpelJob* __restrict__ subOut, MeSearchOut* __restrict__ out) {
  extern __shared__ __align__(16) int16_t sTz[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ji = ctaFirst[blockIdx.x] + warp;
  if (ji >= ctaFirst[blockIdx.x + 1]) return;                          // warp uniform
  const MeTzJob j = jobs[ji];
  const MeSearchCost c = cost[j.outIndex];
  const int w = j.w, nr = (j.h + (1 << j.subShift) - 1) >> j.subShift;
  int16_t* sCur = sTz + warp * maxSamples;
  const int16_t* cur = mp.cur + j.curOff;
  const uint32_t invW = me_inv((uint32_t)w);
  for (int s = lane; s < nr * w; s += 32) {
    const int r = (int)__umulhi((uint32_t)s, invW);
    sCur[s] = cur[(size_t)(r << j.subShift) * mp.curStride + s - r * w];
  }
  __syncwarp();
  const int refStride = mp.refStride[j.refSlot];
  const int16_t* ref0 = mp.ref[j.refSlot] + j.refOff;
  const int G = me_tz_lanes(nr * w), g = lane & (G - 1), slot = lane / G, P = 32 / G;
  const MeTzState st = me_tz_walk(j, c, [&](const MeTzStage& s, MeTzState& state) {
    unsigned long long pend = kMeNoKey;
    for (int base = 0; base < s.n; base += P) {
      const int i = base + slot, end = min(base + P, s.n);
      MeTzPoint q;
      q.ok = false;
      if (i < s.n) q = me_tz_point(s, i);
      uint32_t part = q.ok ? me_tz_sad_part(sCur, ref0 + (long long)q.y * refStride + q.x, refStride, w, nr, j.subShift, g, G) : 0u;
      for (int m = 1; m < G; m <<= 1) part += __shfl_xor_sync(0xffffffffu, part, m);
      const unsigned long long key = q.ok ? ((unsigned long long)me_tz_probe_cost(part, j.subShift, mp.bitDepth, c, q.x, q.y) << 32) | (uint32_t)i : kMeNoKey;
      const int k1 = me_tz_seg_of(s, end - 1);
      for (int k = me_tz_seg_of(s, base); k <= k1; k++) {               // the segments of the chunk, in order
        unsigned long long kk = i < end && me_tz_seg_of(s, i) == k ? key : kMeNoKey;
        for (int m = G; m < 32; m <<= 1) kk = me_key_min(kk, __shfl_xor_sync(0xffffffffu, kk, m));
        pend = me_key_min(pend, kk);
        if (me_tz_seg_first(s, k + 1) <= end) {                          // segment k is complete
          const bool stop = me_tz_fold(state, s, pend);
          pend = kMeNoKey;
          if (stop) return;
        }
      }
    }
  });
  if (lane == 0) me_tz_finish(st, j, c, refStride, subIn, subOut, out);
}

cudaError_t launch_me_tz_search(const MePlanes& mp, const MeTzJob* jobs, const int32_t* ctaFirst, int nCta, int maxSamples, const MeSearchCost* cost,
                                const SubpelJob* subIn, SubpelJob* subDev, const int32_t* fracJob, int nFrac, uint32_t* tables, MeSearchOut* out, cudaStream_t st,
                                int* launches) {
  if (nCta <= 0) return cudaSuccess;
  me_tz_kernel<<<nCta, 32 * kTzWarps, (size_t)kTzWarps * maxSamples * sizeof(int16_t), st>>>(mp, jobs, ctaFirst, maxSamples, cost, subIn, subDev, out);
  if (launches) *launches += 1;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess || nFrac <= 0) return e;
  if ((e = launch_me_subpel(mp, subDev, nFrac, tables, st, launches)) != cudaSuccess) return e;
  me_search_walk_kernel<<<(nFrac + 127) / 128, 128, 0, st>>>(fracJob, nFrac, cost, tables, out);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace cucd
