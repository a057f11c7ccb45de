// nm_sift_internal.cuh -- workspace layout shared by the batched SIFT kernels.
//
// HBM layout (per context, sized for max_batch frames B, see DESIGN.md):
//   per octave o (w_o = width>>o, h_o = height>>o, pitch_o = align32(w_o)):
//     levels  [B][6][h_o][pitch_o] fp32      Gaussian levels (reference PyramidData::_octave)
//     grad    [B][3][h_o][pitch_o] float2    gradient maps   (reference PyramidData::_grad)
//     bitmap  [B][3][h_o][wpr_o]   uint32    1 bit per pixel: accepted keypoint
//     wprefix [B][3][h_o*wpr_o]    int32     exclusive popcount prefix inside the segment
//     need    [B][3][ceil(h_o/8)][wpr_o] u8  gradient blocks (8 rows x 32 columns) read by a keypoint window
//   seg_raw   [B][n_oct*3] int   accepted keypoints per (octave, level) before the
//                                early-return rule
//   seg_cnt   [B][n_oct*3] int   after the rule (siftfunctions.cu:145: levels after the
//                                first empty one in an octave are dropped)
//   seg_off   [B][n_oct*3] int   exclusive offsets in (octave, level) order
//   counts    [B]          int   min(total, capacity)
//   kpts      [B][cap] float4, orient [B][cap] float2, meta [B][cap] int (octave)
//   desc      [B][cap][128] fp32, x,y [B][cap] fp32
#pragma once
#include "nm_common.cuh"

#define NM_MAX_OCTAVES 12

struct NmOctave {
    float*    levels;
    float2*   grad;
    uint32_t* bitmap;
    int*      wprefix;
    int*      cand_n;          // [B * tiles]: candidates of each 32 x 32 tile handed from extrema_kernel to refine_list_kernel
    unsigned short* cand;      // [B * tiles][32]: level << 10 | tile row << 5 | tile column
    unsigned char* need;       // [B][3][ceil(h/8)][wpr]: 8-row x 32-column blocks of the gradient maps that a keypoint window reads
    long long level_elems;     // h*pitch
    int       w, h, pitch, wpr;
    float     xper;
};

struct NmOctaveTable {
    NmOctave o[NM_MAX_OCTAVES];
    int      n_oct;
};

struct NmDetectParams {
    float peak, edge, sigma_0;
    int   num_dogs;
    unsigned long long mask;   // cudaTextureObject_t of the caller's mask (compute_keypoints_with_mask), 0 = none
};

// nm_extrema.cu
struct NmBlurTma;
// TMA descriptor of an octave's level planes for `batch` frames (oc.levels = first frame): box = the
// extrema kernel's 40 x 34 x 6 window.
bool nm_extrema_make_tma(NmBlurTma* t, const NmOctave& oc, int batch);
// extrema + refinement of one octave into NmOctave::bitmap; NM_ERR_UNSUPPORTED without a valid descriptor
int nm_extrema_launch(const NmOctave& oc, const NmDetectParams& dp, int batch, cudaStream_t stream, const NmBlurTma* tma);
// gradient maps of levels 1..3 for all octaves; dense = 0: only the blocks marked in NmOctave::need
int nm_gradmap_launch(const NmOctaveTable& tab, int batch, int dense, cudaStream_t stream);
int nm_rank_launch(const NmOctaveTable& tab, int batch, int* seg_raw, cudaStream_t stream);
int nm_plan_launch(const int* seg_raw, int* seg_cnt, int* seg_off, int* counts, int n_oct, int batch,
                   int capacity, cudaStream_t stream);
// emit: slot <- pixel (x, y, level) of every set bit, in copy_if order; kprefine: slot <- refined keypoint payload
// (one thread per keypoint), which also marks NmOctave::need from the keypoint's windows
int nm_emit_launch(const NmOctave& oc, int octave_index, int n_oct, int batch,
                   const int* seg_cnt, const int* seg_off, int capacity, float4* kpts, int* meta,
                   cudaStream_t stream);
int nm_kprefine_launch(const NmOctaveTable& tab, const NmDetectParams& dp, int batch, int capacity, const int* counts,
                       float4* kpts, const int* meta, cudaStream_t stream);

// nm_orient_desc.cu
int nm_orient_launch(const NmOctaveTable& tab, int batch, int capacity, const int* counts,
                     const float4* kpts, const int* meta, float2* orient, cudaStream_t stream);
int nm_describe_launch(const NmOctaveTable& tab, int batch, int capacity, const int* counts,
                       const float4* kpts, const int* meta, const float2* orient, float* desc,
                       float* x, float* y, int num_dogs, int exact, cudaStream_t stream);
