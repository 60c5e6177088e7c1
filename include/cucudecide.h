/* cucudecide.h - C ABI of libcucudecide.so, the B200 (sm_100a) CU-decision cost engine.
 *
 * Drop-in for the data-parallel cost arithmetic of the HM-16.3 based Fast-CU-Decision-HEVC encoder.
 * The reference has no plugin/FFI layer (its hot path is direct C++ member calls plus the
 * TComRdCost::m_afpDistortFunc table, TComRdCost.h:109), so every entry point names the reference
 * call site (file:line under the reference tree) it replaces.  INTEGRATION.md shows the few lines a
 * maintainer adds to the reference to call them.
 *
 * Conventions
 *   - plain C, no exceptions; every function returns 0 (CUCD_OK) or a negative cucd_status;
 *     cucd_last_error(h) gives the text.  HM's own convention is assert/exit(1)
 *     (CommonDef.h:141-164): the shim turns a non-zero return into FATAL_ERROR_0.
 *   - samples are HM `Pel` = int16_t (TypeDef.h:769) with a caller-given stride in samples; luma only.
 *   - the caller owns every host buffer; the library owns device memory, pinned staging and streams.
 *   - a handle belongs to one encoder instance and one CUDA device.  Every entry point takes the handle's lock, so calls
 *     from several host threads (or from a cucd_queue worker beside the encoder thread) serialise instead of racing;
 *     cucd_last_error / cucd_launch_count / the kernel timers describe the most recent call and are only meaningful to
 *     the thread that made it.  Concurrency across encoder instances = one handle each.
 *   - 8-bit content: samples must lie in 0..255 (bit_depth 8 means exactly that).  The 8-bit kernels carry samples as
 *     bytes; a value outside the range is a caller error and is reduced modulo 256, as storing it into HM's 8-bit
 *     file formats would.  (9/10-bit content: 0..1023.)
 *   - cost tables are uint32_t[35] per PU, index = HEVC intra mode, value = what
 *     distParam.DistFunc returns at TEncSearch.cpp:2339 (Hadamard SATD >> (bitDepth-8)).
 *   - "border" = the unfiltered reference samples of a PU as a linear array of 4N+1 int16:
 *     [0..2N-1] left column from the below-left end up to the top, [2N] the top-left corner,
 *     [2N+1..4N] the above row left to right (row 0 / column 0 of m_piYuvExt[Y][UNFILTERED],
 *     TComPattern.cpp:155-163, re-ordered).
 *   - PU order inside a CTU's 341-entry table: depth-major (64,32,16,8,4), z-order inside a depth
 *     (= HM's absPartIdx order).
 */
#ifndef CUCUDECIDE_H
#define CUCUDECIDE_H
#include <stdint.h>
#include <stddef.h>
#ifdef __cplusplus
extern "C" {
#endif

#define CUCD_NUM_INTRA_MODES 35
#define CUCD_PUS_PER_CTU 341
#define CUCD_ABI_VERSION 5

typedef enum {
  CUCD_OK = 0,
  CUCD_ERR_INVALID = -1,      /* bad argument                                  */
  CUCD_ERR_UNSUPPORTED = -2,  /* e.g. bit depth > 10, CTU size != 64           */
  CUCD_ERR_CUDA = -3,         /* a CUDA call failed; see cucd_last_error       */
  CUCD_ERR_NOMEM = -4,
  CUCD_ERR_NO_DEVICE = -5     /* no usable sm_100 device: there is NO CPU path */
} cucd_status;

typedef struct cucd_handle cucd_handle;

/* replaces nothing 1:1; created where TEncTop::create() builds the encoder (TEncTop.cpp:106) */
typedef struct {
  int width, height;           /* luma picture size, multiples of 8 (min CU size)                 */
  int bit_depth;               /* internal luma bit depth, 8..10                                  */
  int ctu_size;                /* 64                                                              */
  int max_depth;               /* 4: CU 64..8, PU 4x4 through NxN                                 */
  int strong_intra_smoothing;  /* SPS flag (TComPattern.cpp:195)                                  */
  int device;                  /* CUDA device ordinal                                             */
  int max_pictures;            /* pictures one cuCUDecide_frames call may carry (>= 1)            */
  int host_threads;            /* persistent worker threads for the host-side TCM fit, 0 = min(8, hardware concurrency);
                                * several handles / ranks on one host: give each cores / handles                    */
  int auto_pin_host;           /* 1: page-lock (cudaHostRegister) caller planes / output buffers of cuCUDecide_frames on first
                                * sight and keep them registered until cucd_destroy - for callers whose buffers live as long
                                * as the handle (HM's TComPicYuv planes, xMalloc, TComPicYuv.cpp:97).  0: only buffers given to
                                * cucd_pin_host_buffer, or already pinned, take the fast path                        */
} cucd_config;

int cucd_abi_version(void);
int cucd_create(const cucd_config* cfg, cucd_handle** out);
int cucd_destroy(cucd_handle* h);
const char* cucd_last_error(const cucd_handle* h);   /* h may be NULL: error of the last failed create */
/* kernels launched by this handle so far (what bench.py reports as gpu_launches) */
long long cucd_launch_count(const cucd_handle* h);
/* Page-lock a caller buffer for the lifetime of the handle (or until cucd_unpin_host_buffer): HM allocates its picture planes
 * once (TComPicYuv::create, xMalloc, TComPicYuv.cpp:97) and pageable memory costs an extra staging copy inside the driver on
 * every transfer.  Exactly [ptr, ptr + bytes) is registered - give the whole allocation (a plane with its margins), so that
 * every later transfer lies inside it: CUDA rejects transfers of partially registered ranges.  A range that overlaps an
 * earlier one replaces it by the union.  Must be unpinned (or the handle destroyed) before the memory is freed. */
int cucd_pin_host_buffer(cucd_handle* h, const void* ptr, size_t bytes);
int cucd_unpin_host_buffer(cucd_handle* h, const void* ptr);

/* ------------------------------------------------------------------------------------------------
 * S1 + S4 (+ frame-replay S2): one picture, or a batch of pictures.
 * Replaces TEncGOP.cpp:1095-1096 -> TEncSlice::getOutlierWithDCT (TEncSlice.cpp:878-1173), the
 * per-CU OBF block sums of TEncCu.cpp:589-600, TEncCu::updateCtuDataISlice (TEncCu.cpp:1874-1893)
 * and, when rec/rmd_cost are given, the full enumeration of the RMD loop TEncSearch.cpp:2327-2361
 * over all 341 PUs of every CTU with borders taken from `rec` under z-scan availability
 * (replay / throughput mode, SURVEY.md 8d).  Any output pointer may be NULL = not wanted.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int16_t* obf;            /* (W/4)*(H/4), row-major: outlier AC coefficients per 4x4 block (0..15)       */
  int16_t* outlier;        /* W*H, row-major: |kept coefficient| / 100 at its coefficient position        */
  double*  yc;             /* 16: outlier threshold per frequency (index 0 unused)                        */
  int32_t* num_obf[4];     /* depth d: (W/s)*(H/s) with s = 64>>d: Num_OBF of every whole CU              */
  int32_t* n_outlier[4];   /* same shape: N_Outlier                                                       */
  int32_t* ctu_src_had;    /* one per CTU: updateCtuDataISlice's iSumHad                                  */
  uint32_t* rmd_cost;      /* nCtu*341*35: SATD tables; 0xFFFFFFFF for PUs not inside the picture         */
  uint8_t* rmd_cost_packed;/* nCtu*CUCD_PACKED_CTU_BYTES: the same tables, narrowest exact type (see below)*/
  /* narrow, exact variants of obf / outlier (either, both or neither may be given beside the int16 planes): the call is
   * PCIe bound, and both planes fit a byte - an OBF count is 0..15, and an AC coefficient of the 4x4 transform is at
   * most 16 368 in magnitude for bit depths <= 10 (a basis row of g_aiT4 other than the DC row sums to at most 128 on
   * its positive side: 128 * max sample >> shift_1st, then the DC row of the other dimension: * 256 >> 8,
   * TEncSlice.cpp:922-926; the DC coefficient itself is dropped, :987-988), so |coeff| / 100 <= 163 */
  uint8_t* obf_u8;         /* (W/4)*(H/4) */
  uint8_t* outlier_u8;     /* W*H */
} cucd_frame_out;

/* Packed cost table of one CTU.  The numbers are those of rmd_cost in the narrowest exact width per PU size, which more
 * than halves the device-to-host traffic of cuCUDecide_frames - the part of the call that is PCIe bound.  The RMD
 * kernels write this layout directly.
 *   bytes [0, 2940)       uint32[21][35]    PUs 0..20    (64x64, 4 x 32x32, 16 x 16x16)
 *   bytes [2940, 7420)    uint16[64][35]    PUs 21..84   (8x8: SATD <= 32 736); 0xFFFF = PU not inside the picture
 *   bytes [7420, 21980)   256*35 values of 13 bits, little-endian bit stream (value i occupies bits [13 i, 13 i + 13)
 *                         of the region): PUs 85..340 (4x4: SATD <= 8 160 for bit depths <= 10); 0x1FFF = not inside */
#define CUCD_COST_NOT_INSIDE 0xFFFFFFFFu   /* table code: the PU does not lie inside the picture */
#define CUCD_COST_PRUNED     0xFFFFFFFEu   /* table code: fork-aware mode (cucd_set_decision_switches) - the encoder would not evaluate this PU;
                                            * 0xFFFE / 0x1FFE in the narrow regions of the packed table */
#define CUCD_PACKED_WIDE_PUS 21
#define CUCD_PACKED_U16_PUS 64
#define CUCD_PACKED_U16_OFFSET (CUCD_PACKED_WIDE_PUS * 35 * 4)
#define CUCD_PACKED_B13_OFFSET (CUCD_PACKED_U16_OFFSET + CUCD_PACKED_U16_PUS * 35 * 2)
#define CUCD_PACKED_CTU_BYTES (CUCD_PACKED_B13_OFFSET + 256 * 35 * 13 / 8)
/* cost of (pu, mode) from one packed CTU table (host-side helper; the "not inside" codes widen to 0xFFFFFFFF) */
uint32_t cucd_packed_cost(const uint8_t* ctu_table, int pu, int mode);
/* the whole table of one CTU widened to uint32[341][35] */
void cucd_unpack_costs(const uint8_t* ctu_table, uint32_t* cost);

int cuCUDecide_frame(cucd_handle* h, const int16_t* orgY, int strideY, const int16_t* recY, int strideRec, int poc,
                     cucd_frame_out* out);
int cuCUDecide_frames(cucd_handle* h, int nPics, const int16_t* const* orgY, int strideY, const int16_t* const* recY,
                      int strideRec, cucd_frame_out* outs);
/* The same for callers that hold 8-bit content as bytes (the file format of 8-bit YUV; halves the upload).  bit_depth must be 8. */
int cuCUDecide_frames_u8(cucd_handle* h, int nPics, const uint8_t* const* orgY, int strideY, const uint8_t* const* recY,
                         int strideRec, cucd_frame_out* outs);

/* Fork-aware enumeration for the frame calls (cuCUDecide_frame(s)(_u8), cucd_dev_frames*).  The fork's whole point is that on
 * Testing pictures (POC % 60 >= 3, tools_YS.cpp:1237-1242) the per-depth switches set after the verify picture
 * (SetDecisionSwitch, tools_YS.cpp:1123-1154: g_bDecisionSwitch[depth][model][Skip2Nx2N / TerminateCU]) let the Naive model's
 * prediction from Num_OBF (tools_YS.cpp:686-695) skip work in TEncCu::xCompressCU: Skip2Nx2N drops the 2Nx2N intra candidate of
 * a CU with Num_OBF > 0 (TEncCu.cpp:951-996, 1040), TerminateCU stops the recursion (and NxN at depth 3) below a CU with
 * Num_OBF == 0 (:1140-1143, 1257-1260); boundary CUs are never predicted (:488-489, 645).
 * With enable != 0 the frame calls compute Num_OBF first and evaluate only the PUs that recursion still reaches; every other
 * PU inside the picture holds CUCD_COST_PRUNED in all 35 modes.  The caller (the encoder's train / verify / test schedule)
 * switches this on for Testing pictures only and passes the switches it holds; enable = 0 restores the full enumeration. */
int cucd_set_decision_switches(cucd_handle* h, int enable, const uint8_t skip2Nx2N[4], const uint8_t terminateCU[4]);

/* ------------------------------------------------------------------------------------------------
 * S2: intra rough mode decision for a batch of PUs with caller-supplied borders.
 * Replaces the body of the loop TEncSearch.cpp:2327-2361 minus xModeBitsIntra: for PU i,
 * sad[i*35 + m] = predIntraAng(m) + xGetHADs.  PUs may have mixed sizes; org holds the source
 * blocks back to back (N*N each, row-major), border the 4N+1 arrays back to back, in PU order.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  uint8_t log2_size;        /* 2..6 */
  uint8_t reserved[3];
} cucd_pu_desc;
int cucd_intra_rmd_batch(cucd_handle* h, int nPU, const cucd_pu_desc* desc, const int16_t* org, const int16_t* border,
                         uint32_t* sad);

/* ------------------------------------------------------------------------------------------------
 * S2, asynchronous and coalescing, for host THREADS of one process (SURVEY.md 8f.1; encoder PROCESSES use cucd_server,
 * include/cucd_ipc.h).  In the live encoder a PU's border is an intermediate state of the reconstruction, so one encoder
 * instance can only offer the few PUs of its current CU at a time.  Several instances therefore share ONE queue on top of a
 * handle: submit copies the request once, into the pinned arena that is being filled, and returns; a worker thread swaps
 * arenas and runs everything that is pending as one batch (one launch per PU size), after a short batching window
 * (CUCD_QUEUE_WINDOW_US, default 30: the instances released by the previous batch come back within tens of microseconds), and
 * completes the tickets in submission order.  A failed batch fails its own tickets only.  Other calls on `h` from other threads
 * are safe (every entry point takes the handle's lock); they serialise with the worker's batches.
 * ---------------------------------------------------------------------------------------------- */
typedef struct cucd_queue cucd_queue;
int cucd_queue_create(cucd_handle* h, cucd_queue** out);
int cucd_queue_destroy(cucd_queue* q);      /* completes what is pending first */
/* thread-safe, non-blocking; `sad` (nPU*35 uint32, caller-owned) is valid once cucd_queue_wait(q, *ticket) returned CUCD_OK */
int cucd_queue_submit(cucd_queue* q, int nPU, const cucd_pu_desc* desc, const int16_t* org, const int16_t* border, uint32_t* sad,
                      uint64_t* ticket);
int cucd_queue_wait(cucd_queue* q, uint64_t ticket);
/* how well requests coalesce: requests and PUs submitted, batches (cucd_intra_rmd_batch calls) executed so far */
int cucd_queue_stats(cucd_queue* q, long long* requests, long long* pus, long long* batches);

/* ------------------------------------------------------------------------------------------------
 * S3: integer motion estimation.
 * cucd_set_ref_picture  uploads a reconstructed reference plane with its replicated margins
 *                       (TComPicYuv layout: TComPicYuv.cpp:77-101, extendPicBorder :191).
 * cucd_set_cur_picture  uploads the source plane the PUs are cut from.
 * cucd_me_sad_surface   replaces m_cDistParam.DistFunc at TEncSearch.cpp:421 / :3924 for every
 *                       integer mv of a window: out[off_i + (mvy-top)*(right-left+1) + (mvx-left)]
 *                       = xGetSAD*(cur PU, ref + mv) with iSubShift = sub_shift; off_i = sum of the
 *                       previous PUs' window sizes.  The host adds getCost(mv).
 * Precondition (as HM's own planes satisfy): every sample of the planes given to cucd_set_cur_picture / cucd_set_ref_picture lies
 * in [0, 2^bit_depth); the kernels keep 8-bit samples as bytes and sum 9/10-bit samples in packed 16-bit halves.  Source blocks
 * with other values (the bi-predictive search key) go through cucd_me_sad_surface_src / cucd_me_subpel_cost_src below.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y, w, h;            /* PU position and size in luma samples */
  int ref_idx;               /* slot given to cucd_set_ref_picture    */
  int left, right, top, bottom; /* inclusive integer MV window (iSrchRngHorLeft.. of xTZSearch) */
  int sub_shift;             /* DistParam::iSubShift (1 when FEN and rows > 8, TEncSearch.cpp:350-356) */
} cucd_me_desc;
int cucd_set_ref_picture(cucd_handle* h, int ref_idx, const int16_t* recY, int stride, int marginX, int marginY);
int cucd_set_cur_picture(cucd_handle* h, const int16_t* orgY, int stride);
int cucd_me_sad_surface(cucd_handle* h, int nPU, const cucd_me_desc* desc, uint32_t* sadOut);

/* ------------------------------------------------------------------------------------------------
 * Fractional-pel refinement (SURVEY.md 8f.3).  Replaces the arithmetic of xPatternSearchFracDIF (TEncSearch.cpp:4340-4376):
 * xExtDIFUpSamplingH / Q (:5431-5637, the 8-tap interpolation of TComInterpolationFilter.cpp:57-290) and the distortion of
 * every candidate of xPatternRefinement (:808-865, m_cDistParam.DistFunc at :851).  For PU i and its integer MV (the result of
 * the integer search) cost[i*49 + (dy+3)*7 + (dx+3)] = xGetHADs (use_hadamard, HadamardME=1) or xGetSAD between the source block
 * and the reference interpolated at quarter-pel offset (dx, dy), dx, dy = -3..3.  The host walks the 9-point half-pel stage and
 * the 9-point quarter-pel stage over the table and adds getCost(mv) (strict '<' keeps HM's tie-break).  Pictures as in S3
 * (cucd_set_cur_picture / cucd_set_ref_picture; the margins must cover the 8-tap support: 4 samples beyond the moved block).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y, w, h;            /* PU position and size in luma samples; w, h multiples of 4, 4..64 */
  int ref_idx;               /* slot given to cucd_set_ref_picture */
  int mvx, mvy;              /* integer-pel MV the refinement is centred on */
  int use_hadamard;          /* m_pcEncCfg->getUseHADME() && !lossless (TEncSearch.cpp:822) */
} cucd_subpel_desc;
#define CUCD_SUBPEL_POINTS 49
int cucd_me_subpel_cost(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, uint32_t* cost);

/* ------------------------------------------------------------------------------------------------
 * Motion compensation and distortion of inter candidates.  Replaces xGetInterPredictionError (TEncSearch.cpp:2905-2926: the
 * merge candidates of xMergeEstimation) and xGetTemplateCost (AMVP) for luma: candidate i is one PU at one quarter-pel motion
 * of list 0, list 1 or both.  pred receives TComPrediction::motionCompensation's luma prediction (xPredInterUni, or
 * xPredInterBi: two 14-bit list predictions averaged by TComYuv::addAvg before the clip) and dist[i] the DistFunc of that
 * prediction against the source block of cucd_set_cur_picture: xGetHADs (8x8 tiles when w and h are multiples of 8, else 4x4)
 * or xGetSAD with iSubShift = 0, both >> (bitDepth - 8).  The candidates of a PU's merge list go in one call.  Weighted
 * prediction is not covered (callers with WP slices keep their own path).  References are the slots of cucd_set_ref_picture;
 * the 8-tap support of every used list must stay inside the padded plane:
 *   x + (mvx >> 2) - 3 >= -marginX, x + (mvx >> 2) + w + 3 <= W - 1 + marginX, and the same vertically.
 * pred (may be NULL) holds the clipped w x h blocks back to back, row-major, in candidate order.  nPU == 0 is a no-op.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y, w, h;            /* PU position and size in luma samples; w, h multiples of 4, 4..64 (every HEVC PU shape, AMP included) */
  int ref_idx[2];            /* cucd_set_ref_picture slot of the L0 / L1 prediction; -1 = list unused; at least one >= 0 */
  int mvx[2], mvy[2];        /* quarter-pel MV per list (TComMv units), already clipped by the caller as xPredInterUni does (TComDataCU::clipMv) */
  int use_hadamard;          /* m_pcEncCfg->getUseHADME() && !transquant bypass: xGetHADs, else xGetSAD */
} cucd_mc_desc;
int cucd_me_mc_cost(cucd_handle* h, int nPU, const cucd_mc_desc* desc, uint32_t* dist, int16_t* pred);

/* ------------------------------------------------------------------------------------------------
 * Chroma motion compensation and SSE of the same inter candidates: the chroma half of TComPrediction::motionCompensation and the
 * distortion encodeResAndCalcRdInterCU takes of it.  4:2:0 only; chroma samples use the handle's bit_depth.
 * Prediction: the chroma branch of xPredInterBlk with TComInterpolationFilter::m_chromaFilter (4 taps at p - 1 .. p + 2, filterHor /
 * filterVer), for bi the two 14-bit list predictions averaged by TComYuv::addAvg before the clip.  Weighted prediction is not covered.
 * The planes of a reference slot / of the current picture are (W / 2) x (H / 2) samples; margins and stride in chroma samples (HM:
 * the luma margin >> 1).  Set chroma after luma: cucd_set_ref_picture(slot) marks that slot's chroma unset and cucd_set_cur_picture
 * marks the current chroma unset, so that a slot never pairs the luma of one picture with the chroma of another. */
int cucd_set_ref_picture_chroma(cucd_handle* h, int ref_idx, const int16_t* recCb, const int16_t* recCr, int strideC, int marginX, int marginY);
int cucd_set_cur_picture_chroma(cucd_handle* h, const int16_t* orgCb, const int16_t* orgCr, int strideC);
/* desc: the cucd_mc_desc array of cucd_me_mc_cost, unchanged (x, y, w, h the LUMA PU; the chroma block is (x/2, y/2, w/2, h/2), 2..32
 * on a side; mvx / mvy the luma quarter-pel MVs, i.e. eighth-pel chroma MVs: integer part mv >> 3, fraction mv & 7; use_hadamard is
 * ignored).  The 4-tap support of every used list must stay inside the padded chroma plane:
 *   x/2 + (mvx >> 3) - 1 >= -marginX, x/2 + (mvx >> 3) + w/2 + 1 <= W/2 - 1 + marginX, and the same vertically.
 * sse[2 i] / sse[2 i + 1]: the Cb / Cr getDistPart of candidate i, sum ((org - pred)^2 >> 2 (bitDepth - 8)) in uint32, before
 * m_distortionWeight (the convention of the chroma TU calls).  pred (may be NULL): per candidate the clipped Cb block, then the Cr
 * block, (w/2) x (h/2) each, row-major.  Rejects what cucd_me_mc_cost rejects, a slot whose chroma is not set, and a call before
 * cucd_set_cur_picture_chroma.  nPU == 0 is a no-op. */
int cucd_me_mc_chroma(cucd_handle* h, int nPU, const cucd_mc_desc* desc, uint32_t* sse, int16_t* pred);

/* ------------------------------------------------------------------------------------------------
 * The same two searches for a caller-supplied source block ("pattern key") instead of the block of the current picture:
 * what the bi-predictive refinement of xMotionEstimation needs (if (bBi), TEncSearch.cpp:3787-3797, 3826-3849: the key is
 * m_cYuvPredTemp = 2 * org - prediction of the other list, TComYuv::removeHighFreq, so its samples may be negative or exceed
 * the bit depth's range), xPatternSearch (:3886-3943) over the +-bipredSearchRange window and xPatternSearchFracDIF around its
 * result.  src holds the w x h blocks of the PUs back to back (row-major, any int16); x / y of the descriptors still place
 * the PU inside the reference picture.  No cucd_set_cur_picture needed.
 * ---------------------------------------------------------------------------------------------- */
int cucd_me_sad_surface_src(cucd_handle* h, int nPU, const cucd_me_desc* desc, const int16_t* src, uint32_t* sadOut);
int cucd_me_subpel_cost_src(cucd_handle* h, int nPU, const cucd_subpel_desc* desc, const int16_t* src, uint32_t* cost);

/* ------------------------------------------------------------------------------------------------
 * Motion search: HM's full integer search xPatternSearch (TEncSearch.cpp:3886-3943) and, with CUCD_SEARCH_FRAC, the refinement
 * walk of xPatternSearchFracDIF / xPatternRefinement (:4340-4376, :808-865) around its result, one motion vector per PU and
 * reference in one call: what xMotionEstimation runs when !m_iFastSearch || bBi.  Nothing but the result leaves the GPU.
 *   B(v) = xGetComponentBits(v): t = v <= 0 ? (-v << 1) + 1 : v << 1, B = 1 + 2 floor(log2 t).
 *   cost_s(x, y) = (uint32_t)(lambda * (B((x << s) - pred_x) + B((y << s) - pred_y))) >> 16, the product a wrapping 32-bit
 *     unsigned product, as m_uiCost * getBits(x, y) >> 16.
 *   Integer stage: mvy = top..bottom (outer), mvx = left..right (inner), c = SAD(mv) + cost_2(mv) with SAD the cucd_me_sad_surface
 *     entry; the first strict minimum gives (mvx, mvy) and sad = its SAD.
 *   FRAC: T = the 49-entry cucd_me_subpel_cost table at (mvx, mvy), use_hadamard = CUCD_SEARCH_HADAMARD.
 *     H = (0,0),(0,-1),(0,1),(-1,0),(1,0),(-1,-1),(1,-1),(-1,1),(1,1)   (s_acMvRefineH)
 *     Q = (0,0),(0,-1),(0,1),(-1,-1),(1,-1),(-1,0),(1,0),(-1,1),(1,1)   (s_acMvRefineQ)
 *     half stage:    d_i = T[(2 H_i.y + 3) * 7 + 2 H_i.x + 3] + cost_1(2 mv + H_i); the first strict minimum gives hb
 *     quarter stage: d_i = T[(2 hb.y + Q_i.y + 3) * 7 + 2 hb.x + Q_i.x + 3] + cost_0(4 mv + 2 hb + Q_i); the first strict minimum
 *                    gives qb and frac_cost; qmv = 4 mv + 2 hb + qb.
 * These orders and formulas restate HM-16.3; they could not be checked against the HM sources in this repository (the encoder
 * proof checks them where the reference build exists).
 * Rejected with CUCD_ERR_INVALID (the handle stays usable): whatever cucd_me_sad_surface rejects, unknown flags, a pred component
 * outside [-2^15, 2^15 - 1], nPU < 0, NULL pointers; with CUCD_SEARCH_FRAC also h % 4 != 0 and a window whose 8-tap support can
 * leave the padded plane: x + left - 4 < -marginX, x + right + w + 4 > W - 1 + marginX, and the same vertically (HM's clipMv keeps
 * every legal window inside).  A 1x1 window refines a given integer MV.  nPU == 0 is a no-op.
 * cucd_me_search_src takes the PUs' own w x h source blocks back to back (any int16), as cucd_me_sad_surface_src.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y, w, h;                /* PU, as cucd_me_desc */
  int ref_idx;                   /* cucd_set_ref_picture slot */
  int left, right, top, bottom;  /* inclusive integer window = cMvSrchRngLT / RB after xSetSearchRange (already clipped, >> 2) */
  int sub_shift;                 /* integer stage iSubShift, as cucd_me_desc */
  int pred_x, pred_y;            /* m_mvPredictor in quarter pels (TComRdCost::setPredictor), each in [-2^15, 2^15 - 1] */
  uint32_t lambda;               /* m_uiCost after getMotionCost(true, 0, ..) = (UInt)floor(65536.0 * sqrtLambda) */
  int flags;                     /* CUCD_SEARCH_FRAC | CUCD_SEARCH_HADAMARD */
} cucd_search_desc;
#define CUCD_SEARCH_FRAC     1     /* run xPatternSearchFracDIF's walk around the integer result */
#define CUCD_SEARCH_HADAMARD 2     /* sub-pel DistFunc = xGetHADs (getUseHADME() && !lossless), else xGetSAD */
typedef struct {
  int32_t mvx, mvy;              /* integer result of xPatternSearch (integer pels) */
  uint32_t sad;                  /* ruiSAD = the DistFunc value at (mvx, mvy) */
  int32_t qmvx, qmvy;            /* final MV in quarter pels: 4 mv + 2 half + quarter (FRAC), else 4 mv */
  uint32_t frac_cost;            /* FRAC: ruiCost of xPatternSearchFracDIF (distortion + mv cost of the quarter stage's best), else 0 */
} cucd_search_result;
int cucd_me_search(cucd_handle* h, int nPU, const cucd_search_desc* desc, cucd_search_result* out);
int cucd_me_search_src(cucd_handle* h, int nPU, const cucd_search_desc* desc, const int16_t* src, cucd_search_result* out);

/* ------------------------------------------------------------------------------------------------
 * TZ search: HM's xTZSearch integer walk and, with CUCD_SEARCH_FRAC, the refinement walk of cucd_me_search around its result, one
 * motion vector per PU and reference in one call: what xMotionEstimation runs when m_iFastSearch && !bBi (--FastSearch=1).
 * Nothing but the result leaves the GPU.  TZ_SEARCH_CONFIGURATION: iRaster 5, zero-vector test on, first search diamond with
 * stop after 3 rounds, raster on (not always), raster refinement off, star refinement diamond with no stop.
 *   probe(x, y, p, d): c = SAD(x, y) + cost_2(x, y) (SAD and cost_2 as cucd_me_search, including the generic widths' iSubShift 0);
 *     if c < best: best = c, b = (x, y), dist = d, round = 0, pt = p.  win = [left, right] x [top, bottom]; box = the clip box.
 *   1. best = ~0; probe(clamp(pred_x, 4 clip_left, 4 clip_right) >> 2, (the same for y), 0, 0) (arithmetic shift); probe(0, 0, 0, 0);
 *      with CUCD_SEARCH_TZ_2NX2N probe(clamp(mv2n into box), 0, 0) and rwin = (b +- search_range) clamped into box, else rwin = win.
 *   2. first search, c = b: for D = 1, 2, 4, .. <= search_range: Diamond(c, D); break when round >= 3.
 *   3. if dist == 1: dist = 0, TwoPoint.   4. if dist > 5: dist = 5, probe(x, y, 0, 5) for y = rwin.top, +5, .. <= rwin.bottom (outer),
 *      x = rwin.left, +5, .. <= rwin.right (inner).
 *   5. while dist > 0: c = b, dist = 0, pt = 0; Diamond(c, D) for every D = 1, 2, .. <= search_range; if dist == 1: dist = 0 and
 *      TwoPoint when pt != 0.
 *   6. mvx, mvy = b, sad = SAD(b); FRAC: qmv and frac_cost from cucd_me_search's walk at b, else qmv = 4 b, frac_cost = 0.
 *   Diamond(c, D): round += 1, then the points below in this order (p, d), each skipped when it fails its guard: a point left /
 *   right / above / below the centre must satisfy x >= left / x <= right / y >= top / y <= bottom of win.
 *     D = 1:     (cx, cy-1) 2, (cx-1, cy) 4, (cx+1, cy) 5, (cx, cy+1) 7; d = 1.
 *     D = 2..8:  h = D/2: (cx, cy-D) 2 D, (cx-h, cy-h) 1 h, (cx+h, cy-h) 3 h, (cx-D, cy) 4 D, (cx+D, cy) 5 D, (cx-h, cy+h) 6 h,
 *                (cx+h, cy+h) 8 h, (cx, cy+D) 7 D.
 *     D > 8:     q = D/4, p 0, d D: (cx, cy-D), (cx-D, cy), (cx+D, cy), (cx, cy+D), then for k = 1, 2, 3: (cx-qk, cy-D+qk),
 *                (cx+qk, cy-D+qk), (cx-qk, cy+D-qk), (cx+qk, cy+D-qk).
 *   TwoPoint: c = b; the two points of case pt, p 0, d 2, guarded as above: 1 (-1,0) (0,-1); 2 (-1,-1) (1,-1); 3 (0,-1) (1,0);
 *     4 (-1,1) (-1,-1); 5 (1,-1) (1,1); 6 (-1,0) (0,1); 7 (-1,1) (1,1); 8 (1,0) (0,1), offsets from c.
 * These rules restate HM-16.3 (xTZSearch, xTZSearchHelp, xTZ8PointDiamondSearch, xTZ2PointSearch); they are not pinned against the
 * HM sources in this repository.
 * Rejected with CUCD_ERR_INVALID (the handle stays usable): what cucd_me_search rejects about PU, slot, sub_shift, flags (here
 * CUCD_SEARCH_FRAC | CUCD_SEARCH_HADAMARD | CUCD_SEARCH_TZ_2NX2N), predictor and pointers; win empty or not inside box; a box
 * that does not contain (0, 0) or does not fit int16; a box whose blocks leave the padded plane (x + clip_left < -marginX,
 * x + clip_right + w - 1 > W - 1 + marginX, the same vertically; with FRAC the 8-tap support: 4 samples more on each side and one
 * more on the right / bottom, as cucd_me_search); search_range outside [0, 4095]; mv2n outside int16; with FRAC h % 4 != 0.
 * Every probe lies in box, so the box check bounds every read (HM's clipMv area meets it with an 80-sample margin).  nPU == 0 is
 * a no-op.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y, w, h;                /* PU, as cucd_me_desc */
  int ref_idx;                   /* cucd_set_ref_picture slot */
  int left, right, top, bottom;  /* cMvSrchRngLT / RB of xMotionEstimation (xSetSearchRange around the predictor), integer pels */
  int sub_shift;                 /* iSubShift of xTZSearchHelp (FEN and rows > 8), as cucd_me_desc */
  int pred_x, pred_y;            /* m_mvPredictor, quarter pels, each in [-2^15, 2^15 - 1] */
  uint32_t lambda;               /* m_uiCost, as cucd_search_desc */
  int flags;                     /* CUCD_SEARCH_FRAC | CUCD_SEARCH_HADAMARD | CUCD_SEARCH_TZ_2NX2N */
  int search_range;              /* m_iSearchRange: diamond distances 1, 2, 4, .. <= search_range; raster re-centring range */
  int clip_left, clip_right, clip_top, clip_bottom;  /* TComDataCU::clipMv of the PU's CU, integer pels (HM's quarter-pel bounds >> 2) */
  int mv2n_x, mv2n_y;            /* m_integerMv2Nx2N[list][ref], integer pels; a start point when CUCD_SEARCH_TZ_2NX2N */
} cucd_tz_desc;
#define CUCD_SEARCH_TZ_2NX2N 4     /* xTZSearch's pIntegerMv2Nx2NPred: start at mv2n and re-centre the raster window on the best start */
int cucd_me_tz_search(cucd_handle* h, int nPU, const cucd_tz_desc* desc, cucd_search_result* out);

/* ------------------------------------------------------------------------------------------------
 * Intra luma TU coding (SURVEY.md 8f.2): the arithmetic of TEncSearch::xIntraCodingTUBlock (TEncSearch.cpp:1092-1387) for a
 * batch of luma TUs with caller-supplied borders, packed like S2: org holds the N*N source blocks back to back, border
 * the 4N+1 unfiltered reference arrays; coef / level / pred / reco use the layout of org (N*N per TU, row-major; coefficient
 * [v][u] = vertical x horizontal frequency as TCoeff blocks are stored); dist / abs_sum hold one value per TU.
 * The entropy-coupled parts stay with the caller: RDOQ (xRateDistOptQuant), the CABAC bit count, the RD compare.
 *   cucd_intra_tu_forward  initAdiPatternChType smoothing + predIntraAng + residual (:1160-1224) + the transform half of
 *                          TComTrQuant::transformNxN (xT = partial butterflies / 4x4 DST, or xTransformSkip;
 *                          TComTrQuant.cpp:860-919, 1376-1440, 1857-1978): coef = m_plTempCoeff, what xRateDistOptQuant
 *                          reads; pred (may be NULL) = piPred.
 *   cucd_intra_tu_recon    the half after the quantiser for levels chosen by the caller (the host's RDOQ):
 *                          invTransformNxN (xDeQuant + xIT / xITransformSkip, TComTrQuant.cpp:927-985, 1242-1352, 1462-1586),
 *                          reconstruction with clipping (TEncSearch.cpp:1360-1381), SSE getDistPart (:1385-1386).
 *   cucd_intra_tu_code     the whole chain with HM's plain quantiser (encoders run with --RDOQ=0): xQuant with flat scaling
 *                          lists (TComTrQuant.cpp:1126-1240) and, with CUCD_TU_SIGN_HIDING, signBitHidingHDQ (:991-1123);
 *                          level = pcCoeff, abs_sum = uiAbsSum (the CBF), reco, dist as above.
 * Limits: 4:2:0 intra blocks of 4..32 (luma, or chroma with CUCD_TU_CHROMA), flat scaling lists, no transquant bypass / RDPCM / cross-component prediction /
 * extended precision (all off in the BASELINE configurations).
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  uint8_t log2_size;         /* 2..5 */
  uint8_t mode;              /* luma intra mode 0..34 (uiChFinalMode) */
  int8_t  qp;                /* luma: TComDataCU::getQP(0), the QP before the bit-depth offset, 0..51 */
  uint8_t flags;             /* CUCD_TU_TRANSFORM_SKIP | CUCD_TU_CHROMA */
} cucd_tu_desc;
#define CUCD_TU_TRANSFORM_SKIP 1   /* TComDataCU::getTransformSkip, 4x4 blocks only */
#define CUCD_TU_CHROMA 2           /* a Cb / Cr block of a 4:2:0 picture (SURVEY.md 8f.4: estIntraPredChromaQT TEncSearch.cpp:2660 ->
                                    * xRecurIntraChromaCodingQT -> xIntraCodingTUBlock): unfiltered references only
                                    * (TComChromaFormat.h:147-150), no DC / edge filters (TComPrediction.cpp:284, 822), DCT only,
                                    * mode-dependent scan for 4x4 only; mode = uiChFinalMode (DM already resolved to the luma mode),
                                    * qp = the component's mapped QP (QpParam, TComTrQuant.cpp:66-118) minus the bit-depth offset;
                                    * dist is the plain SSE - the caller applies m_distortionWeight (TComRdCost.cpp:447-450) */
/* `flags` argument of cucd_intra_tu_code */
#define CUCD_TU_INTRA_SLICE 1   /* rounding offset 171/512 instead of 85/512 (TComTrQuant.cpp:1206) */
#define CUCD_TU_SIGN_HIDING 2   /* PPS sign_data_hiding_enabled_flag */
int cucd_intra_tu_forward(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border,
                          int32_t* coef, int16_t* pred);
int cucd_intra_tu_recon(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border,
                        const int32_t* level, int16_t* reco, uint32_t* dist);
int cucd_intra_tu_code(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* org, const int16_t* border, int flags,
                       int32_t* level, int16_t* reco, uint32_t* dist, int32_t* abs_sum);

/* ------------------------------------------------------------------------------------------------
 * Inter TU coding: the arithmetic of TEncSearch::xEstimateResidualQT (TEncSearch.cpp, called by
 * encodeResAndCalcRdInterCU for every inter candidate) for the TUs of inter residual quadtrees.  An inter residual does not depend on the
 * reconstruction of the TU before it, so every TU of every RQT depth of a CU, luma and chroma, and the TUs of all merge
 * candidates of a PU can go in one call.  resi holds the residual blocks org - pred (cut by the caller from pcResi; the luma
 * prediction from cucd_me_mc_cost, the chroma one from cucd_me_mc_chroma), N*N per TU back to back in descriptor order; coef / level / rresi use the same
 * layout, dist / dist_zero / abs_sum hold one value per TU.  Descriptors as above with mode = 0; flags CUCD_TU_TRANSFORM_SKIP
 * (4x4 only) and / or CUCD_TU_CHROMA.
 * Precondition: |resi| <= 2^bit_depth - 1, which the difference of two in-range planes satisfies (the forward stages keep
 * int16 intermediates, exact only in that range).
 * Differences from the intra chain: the DCT at every size (TComTU::useDST is intra-only), the diagonal scan for sign hiding
 * (getCoefScanIdx of a non-intra CU, TComDataCU.cpp:3356-3410), the rounding offset 85/512 of xQuant (an inter CU never lies in
 * an I slice, so the call's flags accept CUCD_TU_SIGN_HIDING only), and the back end: the residual is returned, not a
 * reconstruction.
 *   cucd_inter_tu_forward  TComTrQuant::transformNxN (xT / xTransformSkip, TComTrQuant.cpp:860-919, 1376-1440, 1857-1978):
 *                          coef = m_plTempCoeff, what xRateDistOptQuant reads; dist_zero (may be NULL) = nonCoeffDist /
 *                          puiZeroDist of xEstimateResidualQT = getDistPart(0, resi), the distortion of the TU with CBF 0.
 *   cucd_inter_tu_recon    for levels chosen by the caller (the host's RDOQ): invTransformNxN (xDeQuant + xIT /
 *                          xITransformSkip, TComTrQuant.cpp:927-985, 1242-1352, 1462-1586); rresi (may be NULL) = the
 *                          inverse-transformed residual as Pel (clipped to int16, not a reconstruction), dist =
 *                          getDistPart(rresi, resi) (TComRdCost.cpp:433-455) = sum of ((resi - rresi)^2 >> 2(bit_depth - 8))
 *                          accumulated in uint32 with wrap-around as HM's Distortion (UInt).  A TU whose levels are all
 *                          zero gets rresi = 0 and dist == dist_zero.
 *   cucd_inter_tu_code     the whole chain with HM's plain quantiser (--RDOQ=0): xQuant with flat scaling lists
 *                          (TComTrQuant.cpp:1126-1240) and, with CUCD_TU_SIGN_HIDING, signBitHidingHDQ (:991-1123);
 *                          level = pcCoeff, abs_sum (may be NULL) = uiAbsSum (the CBF), rresi, dist, dist_zero (may be NULL) as above.
 * Chroma distortions are returned before m_distortionWeight (TComRdCost.cpp:447-450).  Limits as for the intra calls; no
 * cross-component prediction, RDPCM, transquant bypass or weighted prediction.  nTU == 0 is a no-op.
 * ---------------------------------------------------------------------------------------------- */
int cucd_inter_tu_forward(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi,
                          int32_t* coef, uint32_t* dist_zero);
int cucd_inter_tu_recon(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi,
                        const int32_t* level, int16_t* rresi, uint32_t* dist);
int cucd_inter_tu_code(cucd_handle* h, int nTU, const cucd_tu_desc* desc, const int16_t* resi, int flags,
                       int32_t* level, int16_t* rresi, uint32_t* dist, uint32_t* dist_zero, int32_t* abs_sum);

/* ------------------------------------------------------------------------------------------------
 * CU texture features and AQ activity of the picture given to cucd_set_cur_picture.
 * cucd_tmv_features  replaces getTMVFeature(rpcBestCU) (tools_YS.cpp:1682-1839, call site TEncCu.cpp:1558-1570):
 *                    feat[i*130 + f*26 + k] = m_adFeature[f][k] of CU i - five 3x3 directional planes (original,
 *                    horizontal, vertical, diagonal, anti-diagonal difference), mean and mean absolute deviation
 *                    over whole / halves / triangles / quadrants, as doubles, quirks of the reference included.
 * cucd_aq_activity   replaces TEncPreanalyzer::xPreanalyze (TEncPreanalyzer.cpp:64-139): for AQ layer d (units of
 *                    ctu_size >> d samples, TEncPic.cpp:128-137) activity[d][unit] = TEncQPAdaptationUnit::getActivity()
 *                    in raster order (ceil(W/unit) x ceil(H/unit); activity[d] may be NULL) and
 *                    avg_activity[d] = TEncPicQPAdaptationLayer::getAvgActivity().  max_aq_depth = 1..4.
 * ---------------------------------------------------------------------------------------------- */
typedef struct {
  int x, y;                  /* CU position in luma samples, multiples of the CU size */
  int log2_size;             /* 3..6 */
} cucd_cu_desc;
#define CUCD_TMV_FEATURES (5 * 26)
int cucd_tmv_features(cucd_handle* h, int nCU, const cucd_cu_desc* cus, double* feat);
int cucd_aq_activity(cucd_handle* h, int max_aq_depth, double* const* activity, double* avg_activity);

/* ------------------------------------------------------------------------------------------------
 * Device-resident variants (inputs already in HBM, outputs stay in HBM): what a caller that keeps
 * pictures on the GPU uses, and what bench.py times for the kernel-only figure.  Pointers are
 * device pointers; `stream` is a cudaStream_t (NULL = default stream).  No host synchronisation.
 * ---------------------------------------------------------------------------------------------- */
/* org/rec: nPics planes, picture p at base + p*picStride samples, rows `stride` samples apart.
 * rmd_cost: nPics*nCtu*341*35 uint32. */
int cucd_dev_rmd_frames(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                        const int16_t* d_rec, long long recPicStride, int recStride, uint32_t* d_rmd_cost);
/* pass 1 of the feature path: d_hist = nPics*16*4096 uint32 histograms of |coeff/8| */
int cucd_dev_feature_hist(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                          uint32_t* d_hist);
/* pass 2: d_thr = nPics*16 int32 thresholds (Yc*8); outputs tight per picture as in cucd_frame_out */
int cucd_dev_feature_obf(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                         const int32_t* d_thr, int16_t* d_obf, int16_t* d_outlier, int32_t* const d_num_obf[4],
                         int32_t* const d_n_outlier[4], int32_t* d_ctu_src_had);
/* the whole frame path on device-resident pictures, enqueued on `stream`: feature pass 1, RMD replay,
 * host TCM fit (the only host synchronisation: it waits for the pass-1 histograms), feature pass 2.
 * When both the features and the RMD tables are asked for, the feature kernels run on a high-priority stream of the
 * library beside the RMD kernel (forked from `stream` at entry, joined back into it before the call returns), so work
 * the caller enqueues on `stream` afterwards is ordered after every output.
 * All outputs are device pointers, batch-contiguous (picture p at p * per-picture size), any may be
 * NULL except that d_rec and d_rmd_cost go together.  yc_host: nPics*16 doubles on the host or NULL. */
typedef struct {
  int16_t* obf; int16_t* outlier;
  int32_t* num_obf[4]; int32_t* n_outlier[4];
  int32_t* ctu_src_had;
  uint32_t* rmd_cost;
} cucd_dev_out;
int cucd_dev_frames(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                    const int16_t* d_rec, long long recPicStride, int recStride, const cucd_dev_out* out, double* yc_host);
/* S3 and the fractional-pel refinement with the results left in HBM: d_sad / d_cost are device pointers laid out like sadOut /
 * cost of cucd_me_sad_surface / cucd_me_subpel_cost (pictures through cucd_set_cur_picture / cucd_set_ref_picture as there); the
 * descriptors are host memory and are consumed before the call returns.  Enqueued on `stream`, no wait for the GPU.
 * cucd_set_cur_picture / cucd_set_ref_picture wait for the device-resident ME work still queued before they replace a plane, so a
 * caller may upload the next picture right after enqueueing these calls: the queued work sees the pictures it was enqueued with. */
int cucd_dev_me_sad_surface(cucd_handle* h, void* stream, int nPU, const cucd_me_desc* desc, uint32_t* d_sad);
int cucd_dev_me_subpel_cost(cucd_handle* h, void* stream, int nPU, const cucd_subpel_desc* desc, uint32_t* d_cost);
/* The host fit sits between the two feature passes; the split form lets a caller overlap it with GPU work of its own
 * choice - typically the next batch:   begin(i); end(i-1); begin(i+1); end(i); ...   (at most 2 batches in flight).
 * cucd_dev_frames_begin enqueues feature pass 1 and the RMD kernel and returns without waiting;
 * cucd_dev_frames_end waits for the histograms of the OLDEST batch begun, fits, enqueues pass 2 and joins it into the
 * stream given to begin.  cucd_dev_frames = begin + end. */
int cucd_dev_frames_begin(cucd_handle* h, void* stream, int nPics, const int16_t* d_org, long long orgPicStride, int orgStride,
                          const int16_t* d_rec, long long recPicStride, int recStride, const cucd_dev_out* out, double* yc_host);
int cucd_dev_frames_end(cucd_handle* h);
/* Frame-mode RMD has bit-identical implementations: 0 = integer ALU (prediction and Hadamard butterflies in
 * registers); 1 = tcgen05 tensor cores for the angular predictions and the Hadamard stage (the default): kind::i8 for
 * 8-bit content, kind::f16 with fp32 accumulation (every operand and sum an exactly representable integer) for 9/10-bit
 * content; 2 = the half-precision kernel whatever the bit depth (verification).
 * CUCD_RMD_PATH=alu in the environment at create time selects 0. */
int cucd_set_rmd_path(cucd_handle* h, int path);
/* Device time of the RMD kernel inside the last `nCalls` cucd_dev_frames calls (CUDA events recorded on the
 * caller's stream around that launch; ring of 64).  The stream must have been synchronised.  Returns
 * the number of calls averaged, or a negative status; *avg_ms = mean duration of one launch. */
int cucd_rmd_kernel_time(cucd_handle* h, int nCalls, float* avg_ms);
/* Device time between the first and the last kernel of the most recent batch call on this handle (cucd_intra_rmd_batch,
 * cucd_me_sad_surface, cucd_me_subpel_cost, cucd_me_search, cucd_me_tz_search, cucd_me_mc_cost, cucd_me_mc_chroma, cucd_intra_tu_*, cucd_inter_tu_*, cucd_tmv_features, cucd_aq_activity): CUDA events on
 * the library's stream, host<->device
 * copies outside.  What bench_rows.py reports as the kernel-only figure of those paths.  A call small enough for the
 * zero-copy path (its kernels read and write page-locked host memory; CUCD_DIRECT_LIMIT bytes, 96 KB by default) is not
 * timed: after one, this call fails with CUCD_ERR_INVALID. */
int cucd_last_kernel_time(cucd_handle* h, float* ms);
/* the host-side fit that sits between the two passes (TEncSlice.cpp:291-392): hist = 16*4096 counts
 * of ONE picture, nBlocks = (W/4)*(H/4); writes yc[16] and thr[16] */
int cucd_tcm_fit(const uint32_t* hist, int nBlocks, double* yc, int32_t* thr);

#ifdef __cplusplus
}
#endif
#endif
