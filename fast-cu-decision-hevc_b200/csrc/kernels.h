// kernels.h - launch entry points of the CUDA kernels (internal to libcucudecide.so).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rmd_chunk.cuh"

namespace cucd {

constexpr int kHistBins = 4096;     // |coeff/8| <= 4095 for bit depths <= 12 (see feature_kernels.cu)
constexpr int kHistFreqs = 16;      // index 0 (DC) unused

// ---- intra RMD (rmd_kernels.cu) ---------------------------------------------------------------
cudaError_t launch_rmd_frames(const FrameSource& fs, int nPics, int bitDepth, int strong, cudaStream_t st, int* launches);
// per-device set-up of the kernels that need more than 48 KB of dynamic shared memory (cucd_create, after cudaSetDevice)
cudaError_t configure_rmd_kernels();
cudaError_t configure_rmd_tc2_kernels();
// +-(H8 (x) H8), +-(blockdiag H4 (x) H4) as s8 UMMA operands, 16 KB: B operand of the tensor-core SATD
cudaError_t launch_hadamard_operands(int8_t* dst, cudaStream_t st);
// predictions AND Hadamard on tcgen05 (rmd_tc2_kernels.cu); tabWin / tabN4 = tc2::fill_win_tables / fill_n4_tables uploaded by the caller.
// Two launches on st: the border pre-pass writes the reference arrays of every CTU and depth to `prep` (rmd_tc2_prep_bytes(nPics *
// fs.ctusPerPic) bytes of device scratch, which must not be in use by another launch), then the RMD kernel reads them.
cudaError_t launch_rmd_frames_tc2(const FrameSource& fs, int nPics, int strong, const uint8_t* tabWin, const uint8_t* tabN4, const int8_t* hadamard,
                                  uint8_t* prep, cudaStream_t st, int* launches);
size_t rmd_tc2_prep_bytes(int nCtus);
// the two launches one at a time (profiles/ubench)
cudaError_t launch_rmd_border_prep(const FrameSource& fs, int nPics, int strong, uint8_t* prep, cudaStream_t st, int* launches);
cudaError_t launch_rmd_frame_tc2(const FrameSource& fs, int nPics, int strong, const uint8_t* tabWin, const uint8_t* tabN4, const int8_t* hadamard,
                                 const uint8_t* prep, cudaStream_t st, int* launches);
int rmd_tc2_smem_bytes();
// the same on tcgen05 kind::f16 for 9/10-bit content (rmd_tc3_kernels.cu); tables = tc3::fill_win_tables16 / fill_n4_tables16 / fill_had_tables16
cudaError_t configure_rmd_tc3_kernels();
cudaError_t launch_rmd_frames_tc3(const FrameSource& fs, int nPics, int bitDepth, int strong, const uint8_t* tabWin16, const uint8_t* tabN416,
                                  const uint8_t* hadamard16, cudaStream_t st, int* launches);
int rmd_tc3_smem_bytes();
// the same tensor-core rounds for S2 batches of ONE PU size with caller-supplied borders (8-bit content)
cudaError_t launch_rmd_batch_tc2(int log2n, const BatchSource& bs, int strong, const uint8_t* tabWin, const uint8_t* tabN4, const int8_t* hadamard,
                                 cudaStream_t st, int* launches);
cudaError_t launch_rmd_batch(int log2n, const BatchSource& bs, int bitDepth, int strong, cudaStream_t st, int* launches);

// ---- per-picture texture features (feature_kernels.cu) ----------------------------------------
struct FeaturePlanes {
  const int16_t* org; long long orgPicStride; int orgStride;   // source luma
  int W, H, ctusPerRow, ctusPerPic, bitDepth;
};
// pass 1: 4x4 DCT of every block, histogram of |coeff/8| per AC frequency: hist[pic][16][4096]
cudaError_t launch_feature_hist(const FeaturePlanes& fp, int nPics, uint32_t* hist, cudaStream_t st, int* launches);
// plain device -> (UVA-mapped, pinned) host copy by the SMs: keeps small latency-critical results out of the copy-engine
// queue, which cuCUDecide_frames fills with cost-table downloads
cudaError_t launch_copy_words(const uint32_t* src, uint32_t* dst, size_t nWords, cudaStream_t st, int* launches);
// pass 2: outlier thresholds thr[pic][16] (= Yc*8 as int) -> OBF plane, Outlier plane, per-depth CU sums
struct FeatureOut {
  int16_t* obf; long long obfPicStride;           // [(H/4)][(W/4)] tight
  int16_t* outlier; long long outlierPicStride;   // [H][W] tight
  uint8_t* obf8; uint8_t* outlier8;               // the same planes as bytes (exact, see include/cucudecide.h); any of the four may be null
  int32_t* numObf[4]; int32_t* nOutlier[4];       // per depth: [(H/size)][(W/size)] tight
  long long cuPicStride[4];
};
cudaError_t launch_feature_obf(const FeaturePlanes& fp, int nPics, const int32_t* thr, const FeatureOut& out, cudaStream_t st, int* launches);
// source-only DC-less 8x8 Hadamard cost per CTU: ctuHad[pic][ctusPerPic]
cudaError_t launch_ctu_src_had(const FeaturePlanes& fp, int nPics, int32_t* ctuHad, cudaStream_t st, int* launches);
// Fork-aware enumeration (Testing pictures of the fork's train / verify / test schedule): which of a CTU's 341 PUs the encoder
// would still evaluate once the per-depth Skip2Nx2N / TerminateCU switches act on the Naive model's prediction from Num_OBF
// (TEncCu.cpp:645-675, 951-996, 1040-1079, 1140-1143, 1257-1260; tools_YS.cpp:686-695).  needed[pic][ctu][341]: 1 = evaluate.
struct PruneSwitches { uint8_t skip2Nx2N[4], terminateCU[4]; };
cudaError_t launch_prune_mask(const FeaturePlanes& fp, int nPics, const FeatureOut& sums, PruneSwitches sw, uint8_t* needed, cudaStream_t st, int* launches);
// u8 -> int16 samples behind the upload of 8-bit content held as bytes (cuCUDecide_frames_u8); nSamples % 16 == 0, 16-byte aligned
cudaError_t launch_widen_u8(const uint8_t* src, int16_t* dst, size_t nSamples, cudaStream_t st, int* launches);

// ---- CU texture features and AQ activity (texture_kernels.cu) -----------------------------------
struct TmvCu { int32_t x, y, log2n, pad; };
// feat[cu][5][26] doubles (getTMVFeature, tools_YS.cpp:1682-1839)
cudaError_t launch_tmv_features(const int16_t* org, int stride, const TmvCu* cus, int nCu, double* feat, cudaStream_t st, int* launches);
struct AqLayers { int count, total; int part[4]; int off[5]; };   // layer d: units of part[d] samples, results at out[off[d]..off[d+1])
cudaError_t launch_aq_activity(const int16_t* org, int stride, int W, int H, const AqLayers& layers, double* out, cudaStream_t st, int* launches);

// ---- intra luma TU coding chain (tu_kernels.cu) -------------------------------------------------
struct TuJob {
  int32_t orgOff;      // sample offset of the TU's source block (and of its coef / level / pred / reco blocks)
  int32_t borderOff;   // sample offset of its 4N+1 border
  int32_t outIndex;    // TU index in the caller's order (dist / absSum)
  uint8_t mode, ts;    // intra mode 0..34; bit 0 transform skip, bit 1 chroma block (cucd_tu_desc.flags)
  int8_t qp; uint8_t pad;
};
struct TuBatch {
  const int16_t* org; const int16_t* border; const TuJob* jobs; int count;
  int stage;           // 0 forward only (coef, pred out), 1 whole chain with the plain quantiser, 2 reconstruction from given levels
  int bitDepth, strong, intraSlice, signHiding;
  int32_t* coef;       // stage 0: transform output; stage 1: levels out; stage 2: levels in
  int16_t* pred;       // stage 0 (may be null)
  int16_t* reco; uint32_t* dist; int32_t* absSum;   // stages 1, 2
};
cudaError_t launch_intra_tu(int log2n, const TuBatch& tb, cudaStream_t st, int* launches);

// ---- integer-ME SAD surfaces (me_kernels.cu) ---------------------------------------------------
struct MeJob {
  int32_t curOff;      // sample offset of the PU's top-left inside the current picture plane
  int32_t refOff;      // sample offset of the co-located sample inside the padded reference plane
  int32_t refSlot;     // which resident reference plane
  int16_t w, h;
  int16_t left, right, top, bottom;   // integer MV window, inclusive
  int16_t subShift, pad;
  int64_t outOff;      // offset (in uint32) of this PU's surface inside the output buffer
};
struct MePlanes {
  const int16_t* cur; int curStride;   // curStride == 0: `cur` holds caller-supplied source blocks (w x h each, any int16), MeJob / SubpelJob::curOff their offsets
  const int16_t* const* ref;  // device array of plane origins (sample (0,0) of each padded plane)
  const int32_t* refStride;   // device array
  int bitDepth;
};
struct SubpelJob {
  int32_t curOff;      // PU origin inside the current picture plane
  int32_t refOff;      // the PU origin displaced by the INTEGER mv inside the padded reference plane
  int32_t refSlot;
  int16_t w, h;
  int32_t useHadamard;
};
// out[job][49]: distortion at quarter-pel offsets (dy+3)*7 + (dx+3), dx, dy = -3..3 around the integer mv
cudaError_t launch_me_subpel(const MePlanes& mp, const SubpelJob* jobs, int nJobs, uint32_t* out, cudaStream_t st, int* launches);
cudaError_t launch_me_sad(const MePlanes& mp, const MeJob* jobs, int nJobs, const int32_t* tileJob, const int32_t* tileIdx, int nTilesDy, int nTilesO,
                          uint32_t* out, cudaStream_t st, int* launches);

}  // namespace cucd
