// tu_kernels.cu - the intra luma TU coding chain of TEncSearch::xIntraCodingTUBlock (TEncSearch.cpp:1092-1387) on sm_100a:
//   reference smoothing + predIntraAng (TComPattern.cpp:185-283, TComPrediction.cpp:183-496, 755-841)
//   residual (:1207-1224) -> TComTrQuant::transformNxN: xT = xTrMxN / xTransformSkip (TComTrQuant.cpp:860-919, 1933-1978),
//   plain quantiser xQuant + signBitHidingHDQ (:991-1240, flat scaling lists; RDOQ is CABAC-coupled and stays on the host)
//   -> invTransformNxN: xDeQuant (:1242-1352) + xITrMxN / xITransformSkip (:927-985, 1980-2031)
//   -> reconstruction with clipping (:1360-1381) -> SSE getDistPart / xGetSSE* (TComRdCost.cpp:433-455, 970-1315).
// The INTER instantiation is the same chain for the TUs of an inter residual quadtree (TEncSearch::xEstimateResidualQT): the
// residual org - pred comes from the caller (no border, no prediction), the DCT runs at every size (TComTU::useDST is intra-only),
// sign hiding uses the diagonal scan, and the back end returns the inverse-transformed residual with its SSE against the
// residual (getDistPart(rresi, resi)) and the SSE of the residual alone (the CBF-0 distortion, nonCoeffDist), both in uint32.
//
// One CTA of 256 threads codes a chunk of TUs of ONE size: 1 TU of 32x32 (4 samples per thread) or 16x16, 4 of 8x8, 16 of 4x4
// (one sample per thread).  Everything of a TU lives in shared memory; the partial butterflies of the reference are exact
// integer matrix products, evaluated as such (sum_x T[k][x] * src[x], rounding shift per stage) from the 32-point matrix kept in
// shared memory (the N-point matrices are its sub-sampled rows).  int32 rows are padded by one word so that the column
// accesses of the second stage are bank-conflict free.  Traffic per TU: N*N*2 + (4N+1)*2 bytes in, N*N*(4+2) + 8 bytes out -
// a streaming kernel whose arithmetic (4 N-term dot products per sample) stays far below the HBM time for N <= 32.
#include <cuda_runtime.h>
#include <type_traits>
#include "kernels.h"

namespace cucd {

namespace {

struct ScanTables {
  uint8_t cg[3][16];          // inside a 4x4 coefficient group: scan position -> row*4 + col, for diag / hor / ver
  uint8_t grp[3][4][64];      // [scan][log2(groups per side)] : group scan position -> groupRow * g + groupCol
};
// ScanGenerator::GetNextIndex (TComRom.cpp:69-140)
constexpr void scan_next(int type, int w, int h, int& line, int& col) {
  if (type == 0) {
    if (col == w - 1 || line == 0) { line += col + 1; col = 0; if (line >= h) { col += line - (h - 1); line = h - 1; } }
    else { col++; line--; }
  } else if (type == 1) { if (col == w - 1) { line++; col = 0; } else col++; }
  else { if (line == h - 1) { col++; line = 0; } else line++; }
}
constexpr ScanTables make_scan_tables() {
  ScanTables t{};
  for (int s = 0; s < 3; s++) {
    int l = 0, c = 0;
    for (int p = 0; p < 16; p++) { t.cg[s][p] = (uint8_t)(l * 4 + c); scan_next(s, 4, 4, l, c); }
    for (int lg = 0; lg < 4; lg++) {
      const int g = 1 << lg;
      int gl = 0, gc = 0;
      for (int p = 0; p < g * g; p++) { t.grp[s][lg][p] = (uint8_t)(gl * g + gc); scan_next(s, g, g, gl, gc); }
    }
  }
  return t;
}
constexpr ScanTables kScanHost = make_scan_tables();
__constant__ ScanTables kScan = kScanHost;

// distinct magnitudes of the HEVC 32-point core transform: c[m] ~ 64*sqrt(2)*cos(m*pi/64) (TComRom.cpp:356-460)
__constant__ int8_t kDctC[33] = {64, 90, 90, 90, 89, 88, 87, 85, 83, 82, 80, 78, 75, 73, 70, 67, 64,
                                 61, 57, 54, 50, 46, 43, 38, 36, 31, 25, 22, 18, 13, 9, 4, 0};
__constant__ int8_t kDst4[16] = {29, 55, 74, 84, 74, 74, 0, -74, 84, -29, -74, 55, 55, -84, 74, -29};   // TComRom.cpp:343-349
__constant__ int kQuantScales[6] = {26214, 23302, 20560, 18396, 16384, 14564};                          // TComRom.cpp:328-336
__constant__ int kInvQuantScales[6] = {40, 45, 51, 57, 64, 72};
__constant__ int8_t kAngTable[9] = {0, 2, 5, 9, 13, 17, 21, 26, 32};                                    // TComPrediction.cpp:287-288
__constant__ int16_t kInvAngTable[9] = {0, 4096, 1638, 910, 630, 482, 390, 315, 256};

__device__ __forceinline__ int clip3i(int lo, int hi, int v) { return min(hi, max(lo, v)); }

// TComPattern.cpp:523-548 with m_aucIntraFilter (TComPrediction.cpp:50-67), luma
__device__ __forceinline__ bool tu_use_filtered(int lg, int mode) {
  if (mode == 1) return false;
  const int thr = lg == 2 ? 10 : lg == 3 ? 7 : lg == 4 ? 1 : lg == 5 ? 0 : 10;
  return min(abs(mode - 10), abs(mode - 26)) > thr;
}

// one predicted sample at (row r, col c); b = the border the mode reads (linear 4N+1: left bottom->top, corner, above left->right)
__device__ int tu_predict(const int16_t* b, int n, int lg, int mode, int bitDepth, int r, int c, int dc, bool luma) {
  const int n2 = 2 * n;
  const int16_t* top = b + n2 + 1;
  if (mode == 0) {                                                                                     // TComPrediction.cpp:755-805
    return ((n - 1 - c) * b[n2 - 1 - r] + (c + 1) * top[n] + (n - 1 - r) * top[c] + (r + 1) * b[n2 - 1 - n] + n) >> (lg + 1);
  }
  if (mode == 1) {                                                                                     // :183-222, 818-841
    if (n > 16 || !luma) return dc;                                                                    // xDCPredFiltering: luma only
    if (r == 0 && c == 0) return (top[0] + b[n2 - 1] + 2 * dc + 2) >> 2;
    if (r == 0) return (top[c] + 3 * dc + 2) >> 2;
    if (c == 0) return (b[n2 - 1 - r] + 3 * dc + 2) >> 2;
    return dc;
  }
  const bool vertical = mode >= 18;                                                                    // :278-409
  const int am = vertical ? mode - 26 : 10 - mode;
  const int angle = am < 0 ? -kAngTable[-am] : kAngTable[am];
  const int inv = kInvAngTable[abs(am)];
  const int x = vertical ? c : r, y = vertical ? r : c;            // horizontal modes are predicted transposed (:339-344, 397-408)
  const int sMain = vertical ? 1 : -1;                             // main(i) = b[n2 + sMain*i], side(i) = b[n2 - sMain*i]
  if (angle == 0) {
    int v = b[n2 + sMain * (x + 1)];
    if (x == 0 && n <= 16 && luma) v = clip3i(0, (1 << bitDepth) - 1, v + ((b[n2 - sMain * (y + 1)] - b[n2]) >> 1));      // :356-362
    return v;
  }
  const int delta = (y + 1) * angle, di = delta >> 5, df = delta & 31;
  const int k0 = x + di + 1, k1 = k0 + 1;
  // negative indices are the projected side samples (:300-322): ref[k] = side[(128 + |k| * invAngle) >> 8]
  const int r0 = k0 >= 0 ? b[n2 + sMain * k0] : b[n2 - sMain * ((128 - k0 * inv) >> 8)];
  if (df == 0) return r0;
  const int r1 = k1 >= 0 ? b[n2 + sMain * k1] : b[n2 - sMain * ((128 - k1 * inv) >> 8)];
  return ((32 - df) * r0 + df * r1 + 16) >> 5;
}

}  // namespace

// One 1-D transform stage for the outputs of this thread: acc[i] = sum_x M[o0 + i][x] * in[x].  `in` = the thread's input row as packed
// int16 pairs, `mat` = the stage's matrix as int8 rows of N bytes (MW = N / 4 words): one broadcast LDS.32 + two IDP.2A per 4 terms.
template <int N, int KPT>
__device__ __forceinline__ void tu_matvec(const uint32_t (&in)[N / 2], const uint32_t* __restrict__ mat, int o0, int (&acc)[KPT]) {
  constexpr int MW = N / 4;
#pragma unroll
  for (int i = 0; i < KPT; i++) {
    const uint32_t* m = mat + (o0 + i) * MW;
    int a = 0;
#pragma unroll
    for (int w = 0; w < MW; w++) {
      const int tw = (int)m[w];
      a = __dp2a_lo((int)in[2 * w], tw, a);
      a = __dp2a_hi((int)in[2 * w + 1], tw, a);
    }
    acc[i] = a;
  }
}

template <int LG, bool INTER>
__global__ void __launch_bounds__(256)
tu_kernel(const TuBatch tb) {
  constexpr int N = 1 << LG, NN = N * N, P = N + 1;
  constexpr int TPT = NN < 256 ? NN : 256;       // threads per TU
  constexpr int TUS = 256 / TPT;                 // TUs per CTA
  constexpr int IPT = NN / TPT;                  // samples per thread
  constexpr int CGS = NN / 16;                   // coefficient groups per TU
  constexpr int KG = TPT / N;                    // transform stages: a thread owns input row (t % N) and KPT = N / KG = IPT outputs
  constexpr int PW = N / 2 + 1;                  // words per row of the packed int16 stage arrays (odd: conflict-free row loads)
  constexpr int MW = N / 4;
  __shared__ __align__(16) int8_t sMF[NN], sMI[NN];         // forward matrix [k][x] = T_N[k][x], inverse matrix [x][k] = T_N[k][x]
  __shared__ __align__(16) int8_t sDF[16], sDI[16];          // the 4x4 DST pair (luma 4x4 only)
  __shared__ int16_t sUnf[TUS][4 * N + 2], sFil[TUS][4 * N + 2];
  __shared__ int16_t sPred[TUS][NN];
  __shared__ uint32_t sIn[TUS][N * PW], sMid[TUS][N * PW];   // packed int16 pairs, row-major
  __shared__ int32_t sB[TUS][N * P];                         // transform output / residual, row-padded
  __shared__ int32_t sLevel[TUS][NN], sDelta[TUS][NN];
  __shared__ int sAbs[TUS], sDist[TUS], sCgNz[TUS][CGS];
  __shared__ uint32_t sZero[TUS];                            // INTER: SSE of the residual alone
  using Acc = std::conditional_t<INTER, uint32_t, int>;      // INTER sums wrap as HM's Distortion (UInt) does
  constexpr int SEG = TPT < 32 ? TPT : 32;                   // 4x4 TUs: two per warp, sums reduced inside the TU's 16 lanes

  const int tid = threadIdx.x, grp = tid / TPT, t = tid % TPT;
  const int tuIdx = blockIdx.x * TUS + grp;
  const bool live = tuIdx < tb.count;
  const TuJob job = live ? tb.jobs[tuIdx] : TuJob{0, 0, 0, 0, 0, 0, 0};
  const int bd = tb.bitDepth, mode = job.mode, ts = job.ts & 1;
  const bool luma = !(job.ts & 2);
  const bool dst = !INTER && N == 4 && luma;                 // TComTU::useDST: intra luma 4x4
  const int row = t & (N - 1), kg = t >> LG;                 // transform-stage role of this thread

  for (int i = tid; i < NN; i += 256) {                      // rows of the 32-point matrix, sub-sampled (TComRom.cpp:356-460)
    const int k = i >> LG, x = i & (N - 1);
    int a = (k * (32 >> LG) * (2 * x + 1)) & 127;
    if (a > 64) a = 128 - a;
    const int8_t v = k == 0 ? (int8_t)64 : (a <= 32 ? kDctC[a] : (int8_t)-kDctC[64 - a]);
    sMF[k * N + x] = v; sMI[x * N + k] = v;
  }
  if (!INTER && N == 4 && tid < 16) { sDF[tid] = kDst4[tid]; sDI[(tid & 3) * 4 + (tid >> 2)] = kDst4[tid]; }
  if (!INTER && live) {
    const int16_t* bsrc = tb.border + job.borderOff;
    for (int i = t; i < 4 * N + 1; i += TPT) sUnf[grp][i] = bsrc[i];
  }
  if (t == 0) { sAbs[grp] = 0; sDist[grp] = 0; if (INTER) sZero[grp] = 0; }
  __syncthreads();
  // ---- reference smoothing (TComPattern.cpp:185-283) ----------------------------------------------------------------
  if constexpr (!INTER) {
    const int16_t* b = sUnf[grp];
    bool strong = false;
    if (N == 32 && tb.strong) {
      const int thr = 1 << (bd - 5);
      strong = abs(b[0] + b[2 * N] - 2 * b[N]) < thr && abs(b[2 * N] + b[4 * N] - 2 * b[3 * N]) < thr;
    }
    for (int i = t; i < 4 * N + 1; i += TPT) {
      int v;
      if (i == 0 || i == 4 * N) v = b[i];
      else if (strong) {
        if (i < 2 * N) v = ((2 * N - i) * b[0] + i * b[2 * N] + N) >> (LG + 1);
        else if (i == 2 * N) v = b[i];
        else v = ((4 * N - i) * b[2 * N] + (i - 2 * N) * b[4 * N] + N) >> (LG + 1);
      } else v = (b[i - 1] + 2 * b[i] + b[i + 1] + 2) >> 2;
      sFil[grp][i] = (int16_t)v;
    }
    __syncthreads();
  }
  // ---- prediction, residual (int16, row-major: the input rows of the first transform stage) ----------------------------------
  const int16_t* org = tb.org + job.orgOff;                  // INTER: the caller's residual blocks
  int16_t* in16 = reinterpret_cast<int16_t*>(sIn[grp]);
  int16_t* mid16 = reinterpret_cast<int16_t*>(sMid[grp]);
  if constexpr (INTER) {
    // the residual goes straight into the first stage's rows, a copy into sPred for the SSE after sIn is overwritten; its SSE
    // against zero is nonCoeffDist
    const int sh = (bd - 8) << 1;
    uint32_t zero = 0;
#pragma unroll
    for (int e = 0; e < IPT; e++) {
      const int o = t + e * TPT, r = o >> LG, c = o & (N - 1);
      const int v = live ? org[o] : 0;
      sPred[grp][o] = (int16_t)v;
      in16[r * 2 * PW + c] = (int16_t)v;
      zero += (uint32_t)((v * v) >> sh);
    }
#pragma unroll
    for (int m = SEG / 2; m > 0; m >>= 1) zero += __shfl_xor_sync(0xffffffffu, zero, m);
    if ((t & (SEG - 1)) == 0 && zero) atomicAdd(&sZero[grp], zero);
  } else {
    const int16_t* b = (luma && tu_use_filtered(LG, mode)) ? sFil[grp] : sUnf[grp];      // chroma of 4:2:0: never smoothed
    int dc = 0;
    if (mode == 1) { int s = 0; for (int i = 0; i < N; i++) s += b[2 * N + 1 + i] + b[2 * N - 1 - i]; dc = (s + N) / (2 * N); }
#pragma unroll
    for (int e = 0; e < IPT; e++) {
      const int o = t + e * TPT, r = o >> LG, c = o & (N - 1);
      const int p = live ? tu_predict(b, N, LG, mode, bd, r, c, dc, luma) : 0;
      sPred[grp][o] = (int16_t)p;
      in16[r * 2 * PW + c] = (int16_t)(live ? org[o] - p : 0);
      if (live && tb.stage == 0 && tb.pred) tb.pred[job.orgOff + o] = (int16_t)p;
    }
  }
  __syncthreads();
  const int tshift = 15 - bd - LG;
  const uint32_t* matF = reinterpret_cast<const uint32_t*>(dst ? sDF : sMF);
  const uint32_t* matI = reinterpret_cast<const uint32_t*>(dst ? sDI : sMI);
  if (tb.stage != 2) {
    // ---- forward transform (xTrMxN): tmp[k][j] = (sum_x T[k][x] resi[j][x] + add1) >> shift1, coef[k][j] = (sum_x T[k][x] tmp[j][x] + add2) >> shift2.
    //      Transform skip (xTransformSkip) is elementwise.  TUs of one CTA differ, so every barrier is on a path all threads take. -----
    {
      const int shift1 = LG + bd - 9, add1 = shift1 > 0 ? 1 << (shift1 - 1) : 0;
      uint32_t in[N / 2];
      int acc[IPT];
#pragma unroll
      for (int w = 0; w < N / 2; w++) in[w] = sIn[grp][row * PW + w];
      tu_matvec<N, IPT>(in, matF, kg * IPT, acc);
#pragma unroll
      for (int i = 0; i < IPT; i++) mid16[(kg * IPT + i) * 2 * PW + row] = (int16_t)((acc[i] + add1) >> shift1);      // tmp[k][j]
      __syncthreads();
#pragma unroll
      for (int w = 0; w < N / 2; w++) in[w] = sMid[grp][row * PW + w];
      tu_matvec<N, IPT>(in, matF, kg * IPT, acc);
#pragma unroll
      for (int i = 0; i < IPT; i++) {
        const int k = kg * IPT + i;                                                                        // coef[k][j = row]
        if (!ts) sB[grp][k * P + row] = (acc[i] + (1 << (LG + 5))) >> (LG + 6);
      }
      if (ts) {
#pragma unroll
        for (int e = 0; e < IPT; e++) { const int o = t + e * TPT, r = o >> LG, c = o & (N - 1); sB[grp][r * P + c] = (int)in16[r * 2 * PW + c] << tshift; }
      }
    }
    __syncthreads();
    if (tb.stage == 0) {
      if (live) {
#pragma unroll
        for (int e = 0; e < IPT; e++) { const int o = t + e * TPT; tb.coef[job.orgOff + o] = sB[grp][(o >> LG) * P + (o & (N - 1))]; }
        if (INTER && t == 0 && tb.distZero) tb.distZero[job.outIndex] = sZero[grp];
      }
      return;
    }
    // ---- plain quantiser (xQuant, flat scaling) -----------------------------------------------------------------------
    {
      const int baseQp = job.qp + 6 * (bd - 8), per = baseQp / 6, rem = baseQp - per * 6;
      const int qbits = 14 + per + tshift;
      const long long add = (long long)(tb.intraSlice ? 171 : 85) << (qbits - 9);
      const int scale = kQuantScales[rem];
      int mySum = 0;
#pragma unroll
      for (int e = 0; e < IPT; e++) {
        const int o = t + e * TPT, c = sB[grp][(o >> LG) * P + (o & (N - 1))];
        const long long tl = (long long)abs(c) * scale;
        const int q = (int)((tl + add) >> qbits);
        sDelta[grp][o] = (int)((tl - ((long long)q << qbits)) >> (qbits - 8));
        mySum += q;
        sLevel[grp][o] = clip3i(-32768, 32767, c < 0 ? -q : q);
      }
      if (mySum) atomicAdd(&sAbs[grp], mySum);
    }
    __syncthreads();
    // ---- sign-bit hiding (signBitHidingHDQ): one thread per 4x4 coefficient group ---------------------------------------
    if (tb.signHiding) {
      const int scanIdx = INTER || N > (luma ? 8 : 4) ? 0 : (abs(mode - 26) <= 4 ? 1 : (abs(mode - 10) <= 4 ? 2 : 0));   // TComDataCU.cpp:3356-3410
      constexpr int LGG = LG - 2, G = 1 << LGG;
      int gpos = 0;
      if (t < CGS) {
        gpos = kScan.grp[scanIdx][LGG][t];
        const int base = (gpos / G) * 4 * N + (gpos % G) * 4;
        int nz = 0;
        for (int k = 0; k < 16; k++) { const int cg = kScan.cg[scanIdx][k]; nz |= sLevel[grp][base + (cg >> 2) * N + (cg & 3)] != 0; }
        sCgNz[grp][t] = nz;
      }
      __syncthreads();
      if (t < CGS && sAbs[grp] >= 2 && sCgNz[grp][t]) {
        bool lastCG = true;                                   // the first group with a non-zero level in reverse scan order
        for (int g2 = t + 1; g2 < CGS; g2++) lastCG = lastCG && !sCgNz[grp][g2];
        const int base = (gpos / G) * 4 * N + (gpos % G) * 4;
        int pos[16];
#pragma unroll
        for (int k = 0; k < 16; k++) { const int cg = kScan.cg[scanIdx][k]; pos[k] = base + (cg >> 2) * N + (cg & 3); }
        int32_t* lv = sLevel[grp];
        int firstNZ = 16, lastNZ = -1, sum = 0;
        for (int k = 15; k >= 0; k--) if (lv[pos[k]]) { lastNZ = k; break; }
        for (int k = 0; k < 16; k++) if (lv[pos[k]]) { firstNZ = k; break; }
        for (int k = firstNZ; k <= lastNZ; k++) sum += lv[pos[k]];
        if (lastNZ - firstNZ >= 4) {
          const int signbit = lv[pos[firstNZ]] > 0 ? 0 : 1;
          if (signbit != (sum & 1)) {
            int curCost = 0x7fffffff, minCost = 0x7fffffff, minPos = -1, finalChange = 0, curChange = 0;
            for (int k = lastCG ? lastNZ : 15; k >= 0; k--) {
              const int blk = pos[k];
              const int cf = sB[grp][(blk >> LG) * P + (blk & (N - 1))];
              const int du = sDelta[grp][blk];
              if (lv[blk] != 0) {
                if (du > 0) { curCost = -du; curChange = 1; }
                else if (k == firstNZ && abs(lv[blk]) == 1) curCost = 0x7fffffff;
                else { curCost = du; curChange = -1; }
              } else if (k < firstNZ) {
                if ((cf >= 0 ? 0 : 1) != signbit) curCost = 0x7fffffff;
                else { curCost = -du; curChange = 1; }
              } else { curCost = -du; curChange = 1; }
              if (curCost < minCost) { minCost = curCost; finalChange = curChange; minPos = blk; }
            }
            if (lv[minPos] == 32767 || lv[minPos] == -32768) finalChange = -1;
            const int cf = sB[grp][(minPos >> LG) * P + (minPos & (N - 1))];
            if (cf >= 0) lv[minPos] += finalChange; else lv[minPos] -= finalChange;
          }
        }
      }
      __syncthreads();
    }
  } else {
    // ---- stage 2: levels come from the caller (the host's RDOQ) ------------------------------------------------------
    int mySum = 0;
#pragma unroll
    for (int e = 0; e < IPT; e++) { const int o = t + e * TPT; const int l = live ? tb.coef[job.orgOff + o] : 0; sLevel[grp][o] = l; mySum |= l != 0; }
    if (mySum) atomicOr(&sAbs[grp], 1);
    __syncthreads();
  }
  const bool coded = sAbs[grp] > 0;
  // ---- de-quantisation (xDeQuant, flat scaling).  The coefficient (k, j) goes to row j of the inverse transform's input (int16 after the
  //      clip); a transform-skipped block gets its residual right here (xITransformSkip is elementwise) -----------------------------------
  {
    const int baseQp = job.qp + 6 * (bd - 8), per = baseQp / 6, rem = baseQp - per * 6;
    const int rightShift = 6 - (tshift + per), scale = kInvQuantScales[rem];
    const int bitsIn = min(16, 32 + rightShift - 7);
    const int inMin = -(1 << (bitsIn - 1)), inMax = (1 << (bitsIn - 1)) - 1;
    const int off = tshift == 0 ? 0 : 1 << (tshift - 1);
#pragma unroll
    for (int e = 0; e < IPT; e++) {
      const int o = t + e * TPT, k = o >> LG, j = o & (N - 1);
      const int q = clip3i(inMin, inMax, sLevel[grp][o]);
      int v = rightShift > 0 ? (q * scale + (1 << (rightShift - 1))) >> rightShift : (int)((unsigned)(q * scale) << -rightShift);
      v = coded ? clip3i(-32768, 32767, v) : 0;
      in16[j * 2 * PW + k] = (int16_t)v;
      if (ts) sB[grp][k * P + j] = (int)(int16_t)((v + off) >> tshift);                              // stored as Pel (TComTrQuant.cpp:2007)
    }
  }
  __syncthreads();
  // ---- inverse transform (xITrMxN): tmp[j][x] = clip16((sum_k T[k][x] coef[k][j] + 64) >> 7), resi[y][x] = clip16((sum_k T[k][x] tmp[k][y] + add) >> shift2) ---
  {
    const int shift2 = 20 - bd;
    uint32_t in[N / 2];
    int acc[IPT];
#pragma unroll
    for (int w = 0; w < N / 2; w++) in[w] = sIn[grp][row * PW + w];                                  // row = coefficient column j
    tu_matvec<N, IPT>(in, matI, kg * IPT, acc);
#pragma unroll
    for (int i = 0; i < IPT; i++) mid16[(kg * IPT + i) * 2 * PW + row] = (int16_t)clip3i(-32768, 32767, (acc[i] + 64) >> 7);   // tmp[j][x] stored at [x][j]
    __syncthreads();
#pragma unroll
    for (int w = 0; w < N / 2; w++) in[w] = sMid[grp][row * PW + w];                                 // row = spatial row y, entries over k = j of stage 1
    tu_matvec<N, IPT>(in, matI, kg * IPT, acc);
    if (!ts) {
#pragma unroll
      for (int i = 0; i < IPT; i++) sB[grp][row * P + kg * IPT + i] = clip3i(-32768, 32767, (acc[i] + (1 << (shift2 - 1))) >> shift2);
    }
  }
  __syncthreads();
  // ---- reconstruction (INTER: the residual rresi, Pel-clipped above), SSE, outputs ------------------------------------------------------
  {
    const int sh = (bd - 8) << 1;
    Acc sse = 0;
#pragma unroll
    for (int e = 0; e < IPT; e++) {
      const int o = t + e * TPT;
      const int resi = coded ? sB[grp][(o >> LG) * P + (o & (N - 1))] : 0;
      const int rec = INTER ? resi : clip3i(0, (1 << bd) - 1, sPred[grp][o] + resi);
      if (live) {
        const int d = INTER ? sPred[grp][o] - rec : rec - org[o];   // |d| <= 2^bd - 1 + 2^15: d * d fits int
        sse += (Acc)((d * d) >> sh);
        tb.reco[job.orgOff + o] = (int16_t)rec;
        if (tb.stage == 1) tb.coef[job.orgOff + o] = coded ? sLevel[grp][o] : 0;
      }
    }
#pragma unroll
    for (int m = SEG / 2; m > 0; m >>= 1) sse += __shfl_xor_sync(0xffffffffu, sse, m);
    if ((t & (SEG - 1)) == 0 && sse) atomicAdd(reinterpret_cast<Acc*>(&sDist[grp]), sse);
  }
  __syncthreads();
  if (live && t == 0) {
    tb.dist[job.outIndex] = (uint32_t)sDist[grp];
    if (tb.absSum) tb.absSum[job.outIndex] = sAbs[grp];
    if (INTER && tb.distZero) tb.distZero[job.outIndex] = sZero[grp];
  }
}

template <bool INTER>
static void launch_tu_size(int log2n, const TuBatch& tb, cudaStream_t st) {
  switch (log2n) {
    case 2: tu_kernel<2, INTER><<<(tb.count + 15) / 16, 256, 0, st>>>(tb); break;
    case 3: tu_kernel<3, INTER><<<(tb.count + 3) / 4, 256, 0, st>>>(tb); break;
    case 4: tu_kernel<4, INTER><<<tb.count, 256, 0, st>>>(tb); break;
    case 5: tu_kernel<5, INTER><<<tb.count, 256, 0, st>>>(tb); break;
  }
}

cudaError_t launch_tu(int log2n, const TuBatch& tb, cudaStream_t st, int* launches) {
  if (tb.count <= 0) return cudaSuccess;
  if (log2n < 2 || log2n > 5) return cudaErrorInvalidValue;
  if (tb.inter) launch_tu_size<true>(log2n, tb, st); else launch_tu_size<false>(log2n, tb, st);
  if (launches) *launches += 1;
  return cudaGetLastError();
}

}  // namespace cucd
