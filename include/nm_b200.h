/* nm_b200.h -- the C-ABI of the B200-native NiftyMatch feature pipeline.
 *
 * Plain C: raw device/host pointers, ints, floats; no C++/torch/thrust types.
 * Every entry point returns 0 (NM_OK), a negative NM_ERR_* code, or
 * NM_ERR_CUDA_BASE + cudaError_t; nothing throws or calls exit().  Every entry
 * point enqueues ALL of its work on the given stream (nm_stream_t = cudaStream_t).
 * There is no CPU fallback: without a CUDA device every compute call fails.
 *
 * Each function names the reference interface it replaces
 * (paths relative to the reference's src/ directory).
 */
#ifndef NM_B200_H
#define NM_B200_H

#ifdef __cplusplus
extern "C" {
#endif

typedef void* nm_stream_t;      /* cudaStream_t */

enum {
    NM_OK              = 0,
    NM_ERR_INVALID     = -1,    /* bad argument (null pointer, non-positive size, radius > 45, ...) */
    NM_ERR_ALLOC       = -2,    /* device/host allocation failed */
    NM_ERR_OVERFLOW    = -3,    /* an index would not fit the addressed range */
    NM_ERR_UNSUPPORTED = -4,    /* feature not available in this build / on this device */
    NM_ERR_NO_DEVICE   = -5,    /* no sm_100 CUDA device visible */
    NM_ERR_CUDA_BASE   = 1000   /* NM_ERR_CUDA_BASE + cudaError_t */
};

const char* nm_strerror(int code);
/* Compute capability of the current device (major*10+minor), or a negative error. */
int nm_device_cc(void);
const char* nm_version(void);

/* Self-test: compares the gradient kernels' arithmetic (the CUDA math library's main paths of sqrtf,
 * IEEE division and atan2f inlined behind one range test) bit for bit with the expression on the
 * library routines themselves (gpu/kernels/cudamath.cu:47-52) on n generated (dx, dy) pairs;
 * *mismatches_host must come back 0. */
int nm_selftest_gradient(long long n, unsigned seed, long long* mismatches_host);

/* ------------------------------------------------------------------------ */
/* Parameters: mirror of class SiftParams (gpu/sift/siftparams.h:14-99).     */
/* ------------------------------------------------------------------------ */
typedef struct nm_sift_params {
    int   width, height;
    int   num_octaves;          /* floor(log2(min(w,h)*2/32)), >= 1        (:36) */
    int   num_dog_levels;       /* 3                                          (:31) */
    int   level_max, level_min; /* 4, -1                                   (:34-35) */
    float sigma_d_0, sigma_k, sigma_0, sigma_n;                         /* (:39-41) */
    float base_smooth;          /* sqrt(sigma_0^2 k^(2 level_min) - sigma_n^2) (:47) */
    float sigmas[8];            /* sigma_d_0 * k^i, i = 0..4                  (:50) */
    int   num_sigmas;
    float peak_threshold;       /* 0                                          (:32) */
    float edge_threshold;       /* 10                                         (:32) */
} nm_sift_params;

/* SiftParams(width, height) (siftparams.h:30-51). */
int nm_sift_params_init(nm_sift_params* p, int width, int height);
/* PyramidData::create_kernel_for_sigma (gpu/sift/pyramidata.cu:105-123): host taps,
 * taps_host must hold >= 91 floats; *radius = ceil(4 sigma). */
int nm_gaussian_taps(float sigma, float* taps_host, int* radius);

/* ------------------------------------------------------------------------ */
/* Per-stage operators (device pointers; dense row-major images).            */
/* ------------------------------------------------------------------------ */

/* convolve<float> (gpu/kernels/convolution.h:20; convolution.cu:141-159).
 * result = G_col * (G_row * image), zero padded; bitwise the reference's order of
 * operations.  `buffer` (width*height floats) is only touched when radius > 16. */
int nm_blur_f32(float* result, const float* image, float* buffer, int width, int height,
                const float* taps_dev, int radius, nm_stream_t stream);

/* downsample_by_2<float> (gpu/kernels/downsample.h; downsample.cu:20-29). */
int nm_downsample2_f32(float* result, int result_width, int result_height,
                       const float* source, int source_width, int source_height,
                       nm_stream_t stream);

/* subtract<float> (gpu/kernels/cudamath.h:57; cudamath.cu:57-67): C = A - B. */
int nm_subtract_f32(const float* A, const float* B, float* C, int width, int height,
                    nm_stream_t stream);

/* gradient<float> (gpu/kernels/cudamath.h:72; cudamath.cu:72-79): interior pixels
 * get (0.5*|grad|, angle in [0,2pi]); border pixels are left untouched like the
 * reference.  grad = float2 per pixel. */
int nm_gradient_f32(const float* source, float* grad2, int width, int height,
                    nm_stream_t stream);

/* find_keypoints, unmasked (gpu/kernels/keypoint.h:25; keypoint.cu:240-251), on linear
 * DoG images instead of texture objects.  result4 = dense float4 per pixel; entries of
 * rejected pixels are left untouched (caller pre-fills with -1 like siftfunctions.cu:120). */
int nm_keypoints_dense_f32(const float* dog_cur, const float* dog_down, const float* dog_up,
                           int width, int height, float peak_threshold, float edge_threshold,
                           float xper, float sigma_0, int num_dogs, int level,
                           float* result4, nm_stream_t stream);

/* compute_keypoints_with_mask (gpu/sift/siftfunctions.cu:65-98) without the per-octave cudaArray
 * copies: DoG images stay linear, only the caller's mask is a texture (sampled at
 * ((x+.5)*xper, (y+.5)*xper), pixels with mask < 1 are skipped, keypoint.cu:214).
 * tex_mask = 0 behaves like nm_keypoints_dense_f32. */
int nm_keypoints_dense_masked_f32(const float* dog_cur, const float* dog_down, const float* dog_up,
                                  unsigned long long tex_mask, int width, int height,
                                  float peak_threshold, float edge_threshold, float xper,
                                  float sigma_0, int num_dogs, int level, float* result4,
                                  nm_stream_t stream);

/* find_keypoints on cudaTextureObject_t handles, unmasked and masked
 * (gpu/kernels/keypoint.h:25,52).  mask = 0 selects the unmasked variant. */
int nm_keypoints_dense_tex(unsigned long long tex_cur, unsigned long long tex_mask,
                           unsigned long long tex_down, unsigned long long tex_up,
                           int width, int height, float peak_threshold, float edge_threshold,
                           float xper, float sigma_0, int num_dogs, int level,
                           float* result4, nm_stream_t stream);

/* PyramidData::gpu_collate_keypoints_for_level (gpu/sift/pyramidata.cu:84-91): stable
 * compaction of the float4 entries with w >= 0; *count_dev receives the count (device
 * int).  Also fills orient2_fill (if non-null, >= num_pixels float2) with (-1,-1). */
int nm_collate_f32(const float* dense4, int num_pixels, float* out4, int* count_dev,
                   nm_stream_t stream);

/* detect_orientations (gpu/kernels/orientation.h:19; orientation.cu:219-230).
 * grad2 = the octave's gradient maps, level-major (level * oh*ow + y*ow + x). */
int nm_orientations_f32(const float* kpts4, const float* grad2, int num_pts, int octave_width,
                        int octave_height, float gauss_factor, float xper, float* result2,
                        nm_stream_t stream);

/* compute_sift_descriptors (gpu/kernels/descriptor.h:25; descriptor.cu:243-255). */
int nm_descriptors_f32(const float* kpts4, const float* orient2, const float* grad2, int num_pts,
                       int octave_width, int octave_height, int num_dogs, float xper,
                       float* desc, float* x, float* y, nm_stream_t stream);

/* transpose<float> (gpu/kernels/transpose.h:17; transpose.cu:33-40). */
int nm_transpose_f32(float* odata, const float* idata, int width, int height, nm_stream_t stream);

/* compute_brute_force_distance<float> (gpu/kernels/match.h:19; match.cu:120-135):
 * A_t is dim-major (vector_dim x size_A), result is D^T (size_B x size_A). */
int nm_dist2_f32(const float* A_t, int size_A, const float* B, int size_B, int vector_dim,
                 float* result_t, nm_stream_t stream);

/* get_sift_matches<float> (gpu/kernels/match.h:41; match.cu:141-150). */
int nm_set_matches_f32(const float* distance, int rows, int cols, int buffer_width,
                       int* result, float ambiguity, nm_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Fused matcher (replaces compute_sift_matches, gpu/sift/siftfunctions.h:19; */
/* siftfunctions.cu:15-40) without materialising the distance matrix.          */
/* ------------------------------------------------------------------------ */

/* A: nA x 128, B: nB x 128 fp32 row-major on the device; match_io[nA] in/out with the
 * reference's rule (match.cu:88-116).  The candidate search runs on the tensor cores
 * (tcgen05, fp16 operands); the top candidates are re-ranked with the reference's exact
 * fp32 arithmetic, so indices equal the reference's.  distance (nA*nB floats) may be
 * NULL; when given, the exact fp32 matrix is also written (compat). */
int nm_match_f32(const float* A, int nA, const float* B, int nB, float ambiguity,
                 int* match_io, float* distance, nm_stream_t stream);

/* Per-shard records for a sharded database: rec4[a] = (d1, bits(i1 + index_offset), d2, 0)
 * with exact fp32 distances, reference tie rules.  nB may be 0 (d1 = d2 = +inf marker). */
int nm_match_top2_f32(const float* A, int nA, const float* B, int nB, int index_offset,
                      float* rec4, nm_stream_t stream);

/* Merge n_shards record arrays (shard-major: recs[s*nA + a]) and apply the ratio rule;
 * bit-identical to a single-GPU nm_match_f32 over the concatenated database. */
int nm_match_merge_top2(const float* recs4, int n_shards, int nA, float ambiguity,
                        int* match_io, nm_stream_t stream);
/* The same with shard_stride_rows >= nA rows between the record arrays of consecutive shards (recs[s*stride + a]). */
int nm_match_merge_top2_strided(const float* recs4, int n_shards, long long shard_stride_rows, int nA,
                                float ambiguity, int* match_io, nm_stream_t stream);

/* compute_sift_matches (gpu/sift/siftfunctions.cu:15-40) for every CONSECUTIVE pair of a SIFT batch -- frame p
 * against frame p + 1, p = 0 .. n_frames-2 -- in one launch sequence on the tcgen05 engine with no host
 * synchronisation: every size is read on the device (BASELINE.json configs[4], the mosaicking stream).
 *   desc        [n_frames][capacity][128] floats, the layout of nm_sift_results (capacity a multiple of 256)
 *   counts_dev  [n_frames] descriptors per frame (device memory)
 *   match_out   [n_frames-1][capacity] ints: entry (p, a), a < counts[p], receives the index into frame p + 1 or -1;
 *               like _match_indexes in the reference, an entry whose second distance is <= 0 keeps its value
 *               (match.cu:107), and so do the rows >= counts[p]
 *   rec_out4    optional [n_frames-1][capacity] records (d1, bits(i1), d2, 0) -- exact, as nm_match_top2_f32
 *   fallback_rows_dev  optional device int, incremented per row whose exactness certificate failed (those rows
 *               are scanned exactly inside the same kernel) */
int nm_match_pairs_f32(const float* desc, const int* counts_dev, int n_frames, int capacity, float ambiguity,
                       int* match_out, float* rec_out4, int* fallback_rows_dev, nm_stream_t stream);

/* The SPAN LAYOUT of a window of n frames, 1 <= span <= min(8, n - 1): its links are the pairs (t, t + d), 1 <= d <= span,
 * 0 <= t < n - d, stored d-major -- link (t, d) is row l = sum_{e<d} (n - e) + t, and there are
 * L = span * n - span * (span + 1) / 2 rows.  Rows 0 .. n-2 are the consecutive pairs, in the layout of nm_match_pairs_f32.
 * Correspondence i of a link is (frame t point, frame t + d point); a link's model maps frame t to frame t + d.
 *
 * nm_match_pairs_f32 for every link of the layout: match_out and rec_out4 are [L][capacity], entry (l, a) gets the
 * index into frame t + d.  Link (t, d) is bitwise nm_match_f32(frame t, frame t + d); span 1 is bitwise
 * nm_match_pairs_f32.  Every frame is still packed once; sizes are read on the device and nothing synchronises. */
int nm_match_pairs_span_f32(const float* desc, const int* counts_dev, int n_frames, int capacity, int span, float ambiguity,
                            int* match_out, float* rec_out4, int* fallback_rows_dev, nm_stream_t stream);

/* Which candidate-search engine nm_match_* uses: 0 = exact fp32 SIMT scan,
 * 1 = tcgen05 contraction + fp32 re-rank (default when the device is sm_100). */
int nm_match_set_engine(int engine);
int nm_match_get_engine(void);

/* Diagnostics of the tensor-core engine: records like nm_match_top2_f32 (index_offset 0), and
 * *fallback_rows = number of query rows whose exactness certificate failed and that were
 * re-scanned by the exact fp32 engine (host int; the call synchronises the stream).
 * Optional HOST outputs (may be NULL): the candidate lists of the tensor-core scan,
 * cand_scores/cand_index [n_lists][nA][4] (room for 8 lists), *n_lists, and the power-of-two
 * *scale applied before the fp16 rounding. */
int nm_match_tc_probe(const float* A, int nA, const float* B, int nB, float* rec4,
                      int* fallback_rows, float* cand_scores_host, int* cand_index_host,
                      int* n_lists, float* scale, nm_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Input preprocessing (SURVEY.md 8f rank 2).                                  */
/* ------------------------------------------------------------------------ */

/* cuda_grayscale<float> (gpu/kernels/bgra_2_gray.h; bgra_2_gray.cu:8-29): bgra = width*height uchar4
 * pixels (b, g, r, a), output[i] = (float)(0.07*b + 0.72*g + 0.21*r) as the reference's double expression
 * rounds it.  Device pointers; bgra 4-byte aligned. */
int nm_grayscale_bgra_f32(const void* bgra, float* output, int width, int height, nm_stream_t stream);

/* cuda_extract_channel<float> / cuda_put_channel<float> / cuda_set_alpha_to_const (bgra_2_gray.h; bgra_2_gray.cu:
 * 33-112).  channel 0..3 = b, g, r, a; put_channel on channel 3 writes 255 like the reference. */
int nm_bgra_extract_channel_f32(const void* bgra, float* output, int width, int height, int channel, nm_stream_t stream);
int nm_bgra_put_channel_f32(void* bgra, const float* input, int width, int height, int channel, nm_stream_t stream);
int nm_bgra_set_alpha(void* bgra, int width, int height, unsigned char val, nm_stream_t stream);

/* cuda_cast<float, unsigned char> (gpu/kernels/cast.h; cast.cu:7-39): dst = (max_val != 0 && src >= max_val)
 * ? max_val : (unsigned char)src. */
int nm_cast_f32_u8(const float* src, int cols, int rows, unsigned char* dst, unsigned char max_val,
                   nm_stream_t stream);

/* cuda_undistort (gpu/kernels/undistort.h:29; undistort.cu:6-64): radial distortion map.  camera_matrix =
 * {fx, fy, cx, cy}, distortion_coeffs = {k1, k2, k3}, all device pointers (as in the reference). */
int nm_undistort_map_f32(const float* x, const float* y, int cols, int rows, const float* camera_matrix,
                         const float* distortion_coeffs, float* u, float* v, nm_stream_t stream);

/* resample_undistort (gpu/kernels/resample.h:36; resample.cu:104-117, :235-248): result[i] =
 * tex2D<float>(tex, x[i] + 0.5, y[i] + 0.5) * 255.9999f through the caller's texture object. */
int nm_resample_tex_f32(unsigned long long tex, const float* x, const float* y, int cols, int rows,
                        float* result, nm_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Mosaic rendering (SURVEY.md 8f rank 4): gpu/kernels/resample.h.             */
/* Texture objects are the caller's (the reference's CudaTex2D set-up).        */
/* ------------------------------------------------------------------------ */

/* resample_perspective_transform (resample.h:7; resample.cu:83-102, :119-233): x_pos / y_pos receive the
 * (inverse) perspective map of the pixel grid, result (uchar4) the texture sampled there. */
int nm_resample_perspective_bgra(void* result, unsigned long long tex, int cols, int rows, float* x_pos, float* y_pos,
                                 const float* mat3x3, int inverse, nm_stream_t stream);

/* resample_mask (resample.h:12; resample.cu:67-81, :236-244). */
int nm_resample_mask_tex_u8(unsigned char* result, unsigned long long tex, int cols, int rows, const float* x_pos,
                            const float* y_pos, float threshold, nm_stream_t stream);

/* transform_blend (resample.h:16; resample.cu:7-65, :246-258): warp `frame` by mat3x3 into the canvas at
 * offset (tx, ty), blended by the running weights. */
int nm_transform_blend_bgra(void* canvas, int cw, int ch, unsigned long long frame_tex, int fw, int fh, int nw, int nh,
                            const float* mat3x3, int tx, int ty, unsigned long long mask_tex, float* canvas_wts,
                            unsigned long long frame_wts_tex, nm_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Mosaic of a frame stream: the pairwise homographies of a registered        */
/* stream chained and laid out on a canvas, and a chunk of frames blended in  */
/* one pass over the canvas.  No host synchronisation inside.                 */
/* ------------------------------------------------------------------------ */
typedef struct nm_mosaic_ctx nm_mosaic_ctx;

/* frame_w x frame_h BGRA frames, up to max_frames (<= 1024) per blend call.  mask: frame_w*frame_h bytes, weights:
 * frame_w*frame_h floats, host or device memory; bound as textures with the reference's CudaTex2D settings
 * (cudaArray, linear filter, border addressing, unnormalised coordinates; frame and mask read as normalised floats,
 * weights as elements), like the textures a reference client hands to transform_blend.  The context owns one such
 * frame texture per slot.  Calls on one context are ordered by their stream: use one stream per context. */
int nm_mosaic_create(nm_mosaic_ctx** m, int frame_w, int frame_h, int max_frames, const unsigned char* mask, const float* weights);
int nm_mosaic_destroy(nm_mosaic_ctx* m);

/* Placement, one CTA, fp64.  All pointers are device memory.
 *   H_pairs   [n_frames-1][9] row-major: H[p] maps frame p coordinates to frame p+1 (nm_ransac_batch_f32)
 *   status    [n_frames-1][3] as nm_ransac_batch_f32 writes it, or NULL (every pair valid)
 *   anchor9   G[0] (frame 0 -> mosaic), NULL = identity;  G[p+1] = G[p] . H[p]^-1, where H[p] is replaced by the identity
 *             when status[p*3] == 0 or H[p] is singular or non-finite (flag bit 0 of frame p+1).  After each step G is
 *             divided by the power of two at its largest absolute entry (exact; the blend is scale invariant).
 *   footprint of frame k: the bounding box, floor / ceil, of the sampling box [-1, fw] x [-1, fh] mapped through G[k]
 *             (a bilinear sample with non-zero mask weight comes from inside it); empty, flag bit 1, when a corner has
 *             w <= 0, is non-finite or lies beyond 2^30 pixels
 *   origin2   canvas origin (ox, oy) in mosaic pixels, NULL = the least corner over all non-empty footprints
 *   bounds_out  (ox, oy, width, height): the canvas from that origin that holds every footprint
 *   rects_out [n_frames][4] (tx, ty, nw, nh) in canvas pixels ((0, 0, 0, 0) when empty), 16-byte aligned
 *   mats_out  [n_frames][9] canvas-local -> frame coordinates, G[k]^-1 . T(tx + ox, ty + oy) rounded to float: the
 *             mat3x3 of nm_transform_blend_bgra
 *   flags_out [n_frames];  chain_out  [n_frames][9] doubles, G[k], or NULL */
int nm_mosaic_place_f32(const float* H_pairs, const int* status, int n_frames, int frame_w, int frame_h, const float* anchor9,
                        const int* origin2, float* mats_out, int* rects_out, int* flags_out, int* bounds_out, double* chain_out,
                        nm_stream_t stream);

/* frames_bgra: n_frames x frame_h x frame_w uchar4 on the device (the buffer nm_sift_run_bgra takes), frame size equal to
 * the context's; mats / rects as nm_mosaic_place_f32 writes them (rects 16-byte aligned; a rect with nw or nh <= 0 is
 * empty).  Copies frame i into slot i (one cudaMemcpy2DToArrayAsync each) and blends all n frames in one pass over
 * the cw x ch canvas: bitwise equal to n calls of nm_transform_blend_bgra, in frame order, on the context's textures. */
int nm_mosaic_blend_bgra(nm_mosaic_ctx* m, const void* frames_bgra, int n_frames, int frame_w, int frame_h, const float* mats,
                         const int* rects, void* canvas, int cw, int ch, float* canvas_wts, nm_stream_t stream);

/* The context's texture objects (frame slot i -> frame_tex_host[i], max_frames of them; mask; weights), for callers
 * that drive nm_transform_blend_bgra themselves.  Any output may be NULL. */
int nm_mosaic_textures(nm_mosaic_ctx* m, unsigned long long* frame_tex_host, unsigned long long* mask_tex,
                       unsigned long long* wts_tex);

/* ------------------------------------------------------------------------ */
/* Registration after matching (SURVEY.md 8f rank 1): align_points and the    */
/* three RANSAC estimators of gpu/kernels/ransac.h, Jacobi SVD of svd.cu.      */
/* ------------------------------------------------------------------------ */

/* align_points (gpu/kernels/ransac.h:8; ransac.cu:29-59): correspondence i is
 * (src[i], dst[matches[i]]), or (-1,-1,-1,-1) when matches[i] == -1.  Device pointers. */
int nm_align_points_f32(const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                        float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y,
                        const int* matches, int num_pts, nm_stream_t stream);

/* align_points for every consecutive pair of a SIFT batch (frame p, frame p + 1), sizes read on the device:
 * x, y: [n_frames][capacity] keypoint coordinates (nm_sift_results), matches: [n_frames-1][capacity] indices of
 * nm_match_pairs_f32, counts_dev: [n_frames].  Outputs [n_frames-1][capacity]: correspondence (p, i) =
 * (frame p point i, frame p+1 point matches[p][i]), or (-1,-1,-1,-1) when unmatched or i >= counts[p]. */
int nm_align_pairs_f32(const float* x, const float* y, const int* matches, const int* counts_dev, int n_frames,
                       int capacity, float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y, nm_stream_t stream);

/* nm_align_pairs_f32 for every link of the span layout (see nm_match_pairs_span_f32): matches and the outputs are
 * [L][capacity]; correspondence (l, i) = (frame t point i, frame t + d point matches[l][i]), or (-1,-1,-1,-1) when
 * unmatched or i >= counts[t].  Span 1 is bitwise nm_align_pairs_f32. */
int nm_align_pairs_span_f32(const float* x, const float* y, const int* matches, const int* counts_dev, int n_frames,
                            int capacity, int span, float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y,
                            nm_stream_t stream);

/* Estimator kinds. */
#define NM_RANSAC_TRANSLATION 0   /* 1 correspondence / hypothesis (ransac.cu:467-486) */
#define NM_RANSAC_SIMILARITY  1   /* 2 (ransac.cu:437-464, :322-435) */
#define NM_RANSAC_HOMOGRAPHY  2   /* 4 (ransac.cu:488-520, :84-214) */

/* The hypothesis stage on a caller-supplied index list -- what translation_kernel /
 * similarity_transformation_kernel / homography_kernel compute: rand_list holds 1 / 2 / 4 indices per
 * iteration; homographies[it*9..] and inliers[it] are written for every iteration (0 for an iteration
 * with a repeated index).  inlier rule: squared reprojection error < inlier_threshold over the
 * correspondences with src_x >= 0 (ransac.cu:61-82). */
int nm_ransac_hypotheses_f32(int kind, const float* src_x, const float* src_y, const float* dst_x,
                             const float* dst_y, int num_pts, const int* rand_list, int iterations,
                             float inlier_threshold, float* homographies, int* inliers, nm_stream_t stream);

/* ransac_translation / ransac_similarity / ransac_homography (gpu/kernels/ransac.h:12-22; ransac.cu:
 * 526-694) without their host round trips: valid-index list, index draws (counter-based generator on
 * `seed`: reproducible, where the reference seeds std::mt19937 from std::random_device), hypotheses,
 * scores and the first-maximum selection all run on `stream`.  homography: 9 floats, device.
 * status: 3 ints, device: {1 = model written | 0 = fewer than 2 (homography: 4) valid correspondences,
 * the reference's `return false`, homography untouched; inliers of the chosen model; its iteration}. */
int nm_ransac_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                  int num_pts, float inlier_threshold, int iterations, unsigned long long seed,
                  float* homography, int* status, nm_stream_t stream);


/* nm_ransac_f32 for n_pairs frame pairs in ONE launch sequence (a video stream registers every frame to its
 * successor): pair p reads its correspondences at src_x + p*pair_stride (likewise src_y, dst_x, dst_y),
 * counts[p] of them (device ints, clamped to max_pts; NULL = max_pts for every pair), draws with the seed
 * `seed + p`, and writes homographies[p*9..] and status[p*3..].  Pair p's result equals nm_ransac_f32 on that
 * pair with seed + p.  The hypotheses of all pairs share the grid, so the latency of the per-thread SVD chain is
 * paid once per batch, not once per pair. */
int nm_ransac_batch_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                        long long pair_stride, const int* counts, int max_pts, int n_pairs, float inlier_threshold,
                        int iterations, unsigned long long seed, float* homographies, int* status, nm_stream_t stream);

/* Refit of RANSAC models on their inlier sets, and the inlier masks (no reference counterpart).  Arguments as
 * nm_ransac_batch_f32 (the same correspondence buffers; H_in / status_in as it writes them, status_in NULL = every pair
 * has a model).  Pair p: S0 = the inliers of H_in[p] under the RANSAC rule; round r = 1..rounds fits H_r to S(r-1) by
 * least squares (fp64; translation: mean displacement; similarity: linear in Hartley-normalised coordinates;
 * homography: normalised DLT, then Levenberg-Marquardt on the forward transfer error), rounded to float, and keeps it
 * unless it is degenerate, not finite or has fewer inliers than S(r-1); it stops when the inlier set no longer changes.
 * Sets of no more than 1 / 2 / 4 points are not refitted.  rounds = 0 computes the masks only (H_out = H_in).
 *   H_out      [n_pairs][9], may alias H_in; not written for a pair with status_in[p*3] == 0
 *   status_out [n_pairs][3], may alias status_in: {status_in[p][0], inliers of the returned model, refits kept}; {0, 0, 0}
 *              for a pair without a model.  The layout nm_mosaic_place_f32 reads.
 *   inlier_mask [n_pairs][max_pts] bytes 0 / 1 for the returned model (0 at i >= counts[p]), or NULL.
 * One CTA per pair, no workspace and no host synchronisation (the call can be captured in a CUDA graph); pair p's
 * result is bit-reproducible and does not depend on the other pairs. */
int nm_ransac_refine_batch_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                               long long pair_stride, const int* counts, int max_pts, int n_pairs, float inlier_threshold,
                               const float* H_in, const int* status_in, int rounds,
                               float* H_out, int* status_out, unsigned char* inlier_mask, nm_stream_t stream);

/* Joint adjustment of the chain of a window of n_frames frames registered with skip links (no reference counterpart).
 * The window's L links are in the span layout (nm_match_pairs_span_f32): correspondences, pair_stride, counts (per
 * link, NULL = max_pts) and max_pts as nm_ransac_refine_batch_f32 reads them; H_links [L][9], link_status [L][3] and
 * masks [L][max_pts] as it writes them (RANSAC per d with nm_ransac_batch_f32, then the refit or rounds = 0 for the masks).
 *   Unknowns: G_k maps frame k into frame-0 pixels, G_0 = I; G_k = N^-1 Gn_k N, N centres the frame and scales it by
 *     2 / max(frame_w, frame_h), Gn_k in the family of `kind` (2 / 4 / 8 parameters, homography Gn[8] = 1).  fp64.
 *   Initial poses: for k = 1 .. n-1 the smallest d <= span with frame k-d connected, link_status[(k-d, d)][0] == 1 and
 *     at least 1 / 2 / 4 mask points gives G_k = G_(k-d) . H^-1 (the chaining rule of nm_mosaic_place_f32); without one
 *     frame k is disconnected: G_k = G_(k-1), fixed, and its links are ignored.
 *   Cost (nm_ransac_adjust_chain_f32: NM_ADJUST_MOSAIC): sum over the links usable that way (both frames connected)
 *     and their mask points of |pi(G_t s_i) - pi(G_(t+d) d_i)|^2, in frame-0 pixels.
 *   Solver: Levenberg-Marquardt, lambda0 = 1e-3 max diag(J^T J), / 10 after an accepted step, * 10 after a rejected one,
 *     at most `iterations` (>= 1) builds of the banded normal equations, banded Cholesky in one CTA; the final cost is
 *     never above the initial one.
 *   H_out [n-1][9] (may alias H_links): G_(p+1)^-1 G_p rounded to float, divided by its [8], when frame p+1 is connected
 *     (a disconnected frame p gives the pair out of it that reproduces G_(p+1) in nm_mosaic_place_f32), else H_links[p].
 *   status_out [n-1][3] (may alias link_status): {1, inliers of H_out[p] under the RANSAC rule on link (p, 1), LM steps
 *     accepted} for a connected frame p+1, {0, 0, 0} for a disconnected one.
 *   chain_out [n][9] doubles G_k, or NULL;  report_out [4] doubles, or NULL: mean squared residual (px^2) before and
 *     after, residual points, links used.
 * Limits n_frames <= 1024, span <= 8, span < n_frames.  Stream-ordered workspace, no host synchronisation (the call can
 * be captured in a CUDA graph); the result is bit-reproducible. */
int nm_ransac_adjust_chain_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                               long long pair_stride, const int* counts, int max_pts, float inlier_threshold,
                               int n_frames, int span, int frame_w, int frame_h, const unsigned char* masks,
                               const float* H_links, const int* link_status, int iterations, float* H_out,
                               int* status_out, double* chain_out, double* report_out, nm_stream_t stream);

/* Residual of the chain adjustment (nm_ransac_adjust_chain_cost_f32). */
#define NM_ADJUST_MOSAIC   0   /* pi(G_t s_i) - pi(G_(t+d) d_i), frame-0 (mosaic) pixels: nm_ransac_adjust_chain_f32 */
#define NM_ADJUST_TRANSFER 1   /* pi(G_(t+d)^-1 G_t s_i) - d_i, pixels of frame t + d (the RANSAC rule's direction) */

/* nm_ransac_adjust_chain_f32 with a choice of residual; cost NM_ADJUST_MOSAIC is bitwise nm_ransac_adjust_chain_f32.
 * NM_ADJUST_TRANSFER measures every link's residual in the pixels of its own target frame t + d, so it depends only on
 * the relative poses G_(t+d)^-1 G_t: unlike the mosaic cost it gains nothing from shrinking the frames far from frame 0,
 * which on long windows of similarity or homography models contracts the chain.  Unknowns, gauge, initial poses, links
 * used, solver and outputs are those of nm_ransac_adjust_chain_f32; report_out is in pixels of the target frames.  A point
 * with a non-positive third coordinate of G_(t+d)^-1 G_t s_i, or a non-finite residual, makes the cost of a trial point
 * +inf (the step is rejected); at the initial poses it leaves the window unadjusted (initial chain, 0 LM steps, both
 * costs in report_out +inf).  cost outside {NM_ADJUST_MOSAIC, NM_ADJUST_TRANSFER}: NM_ERR_INVALID. */
int nm_ransac_adjust_chain_cost_f32(int kind, int cost, const float* src_x, const float* src_y, const float* dst_x,
                                    const float* dst_y, long long pair_stride, const int* counts, int max_pts,
                                    float inlier_threshold, int n_frames, int span, int frame_w, int frame_h,
                                    const unsigned char* masks, const float* H_links, const int* link_status, int iterations,
                                    float* H_out, int* status_out, double* chain_out, double* report_out, nm_stream_t stream);

/* nm_ransac_adjust_chain_cost_f32 with the poses of frames 0 .. n_fixed-1 held fixed, 1 <= n_fixed <= n_frames - 1: a
 * window that overlaps the end of an adjusted one is adjusted against that one's poses, so the links that cross the
 * window boundary are used, and a live session can append frames to a chain it has already shown.
 *   fixed_chain [n_fixed][9] device doubles: row j maps frame j into any common frame (for example chain_out rows of the
 *     previous window, chain_out + (n_prev - n_fixed) * 9).  It is rebased on the device: F_j = C_0^-1 C_j, renormalised.
 *   fixed_conn [n_fixed] device ints, or NULL = all connected; entry 0 is ignored (frame 0 is the gauge).  A fixed frame
 *     j >= 1 is fixed and disconnected (its links unused, G_j = G_(j-1)) when fixed_conn[j] == 0, when F_j is not finite,
 *     or when C_0 is not finite or singular (|det| <= 1e-12 max|C_0|^3).  With n_fixed == 1 neither array is read.
 *   Initial poses: fixed frames take F_j; a free frame k >= n_fixed takes the rule of nm_ransac_adjust_chain_f32 (frame
 *     k - d may be a fixed frame).  Links used: that rule, and the later frame t + d must be free (a link between two
 *     fixed frames is constant).  Unknowns: the connected free frames; the rows of a fixed frame are the identity with
 *     zero right-hand side, like those of a disconnected frame, and lambda0 is taken over the free rows.
 *   Outputs as nm_ransac_adjust_chain_cost_f32 for every pair and frame: pairs inside the fixed part come from the fixed
 *     poses, chain_out of a connected fixed frame is F_j up to the rounding of the parameter round trip, and the report
 *     covers the links used.
 * n_fixed < 1, n_fixed >= n_frames, or fixed_chain NULL with n_fixed > 1: NM_ERR_INVALID.  No host synchronisation (the
 * call can be captured in a CUDA graph), bit-reproducible; nm_ransac_adjust_chain_cost_f32 is n_fixed = 1 of it. */
int nm_ransac_adjust_chain_fixed_f32(int kind, int cost, const float* src_x, const float* src_y, const float* dst_x,
                                     const float* dst_y, long long pair_stride, const int* counts, int max_pts,
                                     float inlier_threshold, int n_frames, int span, int frame_w, int frame_h,
                                     const unsigned char* masks, const float* H_links, const int* link_status, int n_fixed,
                                     const double* fixed_chain, const int* fixed_conn, int iterations, float* H_out,
                                     int* status_out, double* chain_out, double* report_out, nm_stream_t stream);

/* ------------------------------------------------------------------------ */
/* Batched SIFT detect+describe: the client loop of the reference             */
/* (compute_dog/_gradients/_keypoints/_orientations/_descriptors,             */
/* gpu/sift/siftfunctions.h:30-101, driven per octave) for a batch of frames, */
/* without host synchronisation inside.                                       */
/* ------------------------------------------------------------------------ */
typedef struct nm_sift_ctx nm_sift_ctx;

/* capacity = descriptor slots per frame (SiftData capacity, gpu/sift/siftdata.h:15). */
int nm_sift_create(nm_sift_ctx** ctx, const nm_sift_params* params, int max_batch, int capacity);
int nm_sift_destroy(nm_sift_ctx* ctx);

/* frames_dev: n_frames dense width*height fp32 images on the device.  Results stay in
 * the context's device buffers (accessors below). */
int nm_sift_run(nm_sift_ctx* ctx, const float* frames_dev, int n_frames, nm_stream_t stream);
/* The same on BGRA video frames (n_frames x height x width uchar4, device): the grey conversion of
 * cuda_grayscale<float> is fused into the base blur (the BGRA words are staged by TMA and converted in
 * shared memory), so no grey frame is written to HBM; launches too small for that kernel convert through
 * the context's staging buffer first.  Results equal nm_grayscale_bgra_f32 followed by nm_sift_run. */
int nm_sift_run_bgra(nm_sift_ctx* ctx, const void* frames_bgra_dev, int n_frames, nm_stream_t stream);

/* End-to-end: frames in (pinned or pageable) HOST memory; copies H2D, runs, and copies
 * counts[n_frames], desc[n_frames*capacity*128], x/y[n_frames*capacity] back to the host
 * (any of desc/x/y may be NULL).  Synchronises the stream before returning. */
int nm_sift_run_host(nm_sift_ctx* ctx, const float* frames_host, int n_frames,
                     int* counts_host, float* desc_host, float* x_host, float* y_host,
                     nm_stream_t stream);

/* compute_keypoints_with_mask (gpu/sift/siftfunctions.h:49-57; siftfunctions.cu:65-98) for the batched
 * path: tex_mask = the caller's cudaTextureObject_t, sampled at ((x+.5)*xper, (y+.5)*xper) in every octave;
 * pixels whose sample is < 1 produce no keypoint (gpu/kernels/keypoint.cu:214).  0 = unmasked (default).
 * The texture must outlive the runs that use it. */
int nm_sift_set_mask(nm_sift_ctx* ctx, unsigned long long tex_mask);
/* Convenience for callers without a texture: binds a width x height float mask image (host or device
 * memory) as a cudaArray texture with the reference's CudaTex2D settings (gpu/utils/cudatex2D.cu:12-19:
 * border addressing, linear filter, unnormalised coordinates; element-type reads).  Owned by the context. */
int nm_sift_set_mask_image(nm_sift_ctx* ctx, const float* mask, int width, int height);

/* Device-side results of the last run (valid until the next run / destroy).
 * desc: [max_batch][capacity][128]; x, y: [max_batch][capacity]; kpts4/orient2 likewise;
 * counts: [max_batch] descriptors per frame; seg_counts: [max_batch][num_octaves*3]
 * collated keypoints per (octave, level) after the early-return rule
 * (siftfunctions.cu:145,160). */
int nm_sift_results(nm_sift_ctx* ctx, const float** desc, const float** x, const float** y,
                    const int** counts, const float** kpts4, const float** orient2,
                    const int** seg_counts);
/* Pyramid level `level` (0..5) of `octave` for `frame`: pointer, pitch (floats), w, h. */
int nm_sift_level(nm_sift_ctx* ctx, int frame, int octave, int level, const float** ptr,
                  int* pitch, int* w, int* h);
/* Gradient map (float2) of DoG level `level` (0..2) of `octave` for `frame`.  By default only the 8-row x
 * 32-column blocks that an orientation / descriptor window of an emitted keypoint reads are computed (the
 * reference's compute_gradients, siftfunctions.cu:53-63, fills whole maps; their other pixels are never read
 * by compute_orientations / compute_descriptors); call nm_sift_set_dense_gradients(ctx, 1) before a run
 * whose whole maps are to be read. */
int nm_sift_grad(nm_sift_ctx* ctx, int frame, int octave, int level, const float** ptr2,
                 int* pitch, int* w, int* h);
/* Number of kernels the last nm_sift_run enqueued (for launch accounting). */
int nm_sift_last_launches(nm_sift_ctx* ctx);
/* Stage timing of the next run: when enabled, nm_sift_run records CUDA events around
 * the stages and nm_sift_stage_ms returns {pyramid, extrema+gradient, compaction,
 * orientation, descriptor, total} in milliseconds after synchronising. */
int nm_sift_enable_timing(nm_sift_ctx* ctx, int enable);
/* Descriptor arithmetic: 0 (default) = fp32 evaluation of the reference formulas,
 * 1 = the reference's mixed fp64/fp32 expression shapes (validation mode). */
int nm_sift_set_exact_descriptor(nm_sift_ctx* ctx, int exact);
int nm_sift_stage_ms(nm_sift_ctx* ctx, float* ms6);
/* {pyramid, extrema, compaction, gradient maps, orientation, descriptor, total} of the last timed run. */
int nm_sift_stage_ms7(nm_sift_ctx* ctx, float* ms7);
/* 1 = gradient maps of every pixel (see nm_sift_grad); 0 (default) = only where keypoint windows read. */
int nm_sift_set_dense_gradients(nm_sift_ctx* ctx, int dense);

#ifdef __cplusplus
}
#endif
#endif /* NM_B200_H */
