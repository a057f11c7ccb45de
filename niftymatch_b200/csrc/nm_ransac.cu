// nm_ransac.cu -- frame-to-frame registration after matching (SURVEY.md 8f rank 1).
//
// Replaces the reference's align_points / ransac_translation / ransac_similarity / ransac_homography
// (gpu/kernels/ransac.cu:50-59, :526-694) and the one-sided Jacobi SVD they call (gpu/kernels/svd.cu:
// 200-360, the reference's port of GSL's gsl_linalg_SV_decomp_jacobi).
//
// Provenance note: the reference's svd.cu carries a GNU GPL header of its own (svd.cu:1-20, derived from GSL),
// unlike the rest of the reference.  jacobi_right_vectors below is a restructured restatement of that published
// algorithm (fused dot / norm loop, lane-interleaved shared-memory matrices, templated sizes, no singular-value
// tail), but it follows the same order of operations -- bitwise hypotheses require it -- so whoever ships this
// file should treat it under the terms that apply to svd.cu.
//
// What is kept: the arithmetic of a hypothesis (normalised 4-point DLT / 2-point similarity / 1-point
// translation, Jacobi sweeps with GSL's error-estimate skip rule, the expanded de-normalisation) in the
// reference's order of operations, the inlier rule (squared reprojection error < threshold over the
// correspondences whose src_x >= 0), "first maximum wins", duplicate index draws score 0 with H = 0.
//
// What is different (B200 design):
//  * the reference copies src_x to the HOST, filters the valid indices there, draws the random list with
//    std::mt19937 seeded from std::random_device (not reproducible) and copies it back: three blocking
//    transfers per call.  Here the valid-index compaction, a counter-based generator (splitmix64 of
//    (seed, draw)), the hypotheses, the scores and the arg-max all run on the caller's stream with no host
//    synchronisation; the seed is a parameter, so a run is reproducible;
//  * the reference scores with one thread per hypothesis looping over every correspondence in global
//    memory; here a CTA stages a block of correspondences in shared memory once and each of its threads
//    scores one hypothesis against it (grid = hypothesis blocks x correspondence blocks, integer atomics,
//    so the counts are exact and order independent);
//  * nm_ransac_batch_f32 estimates many frame pairs in one launch sequence (every kernel indexes the pair by a
//    grid dimension): a hypothesis is a long dependent chain (5-9 Jacobi sweeps of 36 rotations, ~1 ms), so
//    one pair at a time leaves the GPU idle; 64 pairs cost 43 us each;
//  * nm_ransac_hypotheses_f32 takes the caller's index list: that is the entry the parity tests drive with
//    the list they also hand to the reference's own kernels (homographies and inlier counts are bitwise the
//    reference's on the same lists, tests/test_gpu_ransac.py).
#include "nm_chain.cuh"

namespace {

constexpr float kEps = 1.1920928955078125e-07f;      // svd.cu:33 (FLT_EPSILON)

// ---- one-sided Jacobi SVD ---------------------------------------------------------------------------
// svd.cu:133-157
__device__ float hyp(float x, float y)
{
    const float xa = fabsf(x), ya = fabsf(y);
    const float mn = fminf(xa, ya), mx = fmaxf(xa, ya);
    if (mn == 0.f) return mx;
    const float u = mn / mx;
    return mx * sqrtf(1.f + u * u);
}

// A thread's matrix lives in shared memory, element e of lane l at [e * kHypThreads + l]: dynamic column
// indices (j, k) would put a thread-local array in local memory; this layout is bank-conflict free and the
// rotations read and write it at shared-memory latency.
constexpr int kHypThreads = 32;
struct SMat {
    float* p;
    __device__ __forceinline__ float& operator[](int e) const { return p[e * kHypThreads]; }
};

// Right singular vectors Q (COLS x COLS) of A (ROWS x COLS, destroyed); svd.cu:200-316.  The singular
// values and the column normalisation of A that follow in the reference (:318-352) are not read by any
// caller and are not computed.  err: COLS column error estimates (the reference's S).
template <int ROWS, int COLS>
__device__ void jacobi_right_vectors(SMat A, SMat Q, SMat err)
{
    const float tol = (float)(10 * ROWS) * kEps;
    const int sweepmax = 5 * COLS > 12 ? 5 * COLS : 12;
    for (int i = 0; i < COLS * COLS; ++i) Q[i] = 0.f;
    for (int i = 0; i < COLS; ++i) Q[i * COLS + i] = 1.f;
    for (int j = 0; j < COLS; ++j) {
        // dnrm2 (svd.cu:159-198)
        float scale = 0.f, ssq = 1.f;
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
            const float x = A[i * COLS + j];
            if (x != 0.f) {
                const float ax = fabsf(x);
                if (scale < ax) { ssq = 1.f + ssq * (scale / ax) * (scale / ax); scale = ax; }
                else ssq += (ax / scale) * (ax / scale);
            }
        }
        err[j] = kEps * (scale * sqrtf(ssq));
    }
    int count = 1, sweep = 0;
    while (count > 0 && sweep <= sweepmax) {
        count = COLS * (COLS - 1) / 2;
#pragma unroll 1
        for (int j = 0; j < COLS - 1; ++j)
#pragma unroll 1
            for (int k = j + 1; k < COLS; ++k) {
                // dot product and the two scaled norms in ONE pass over the rows: three independent dependency
                // chains in flight instead of three loops back to back (each quantity sees the operations of
                // ddot / dnrm2, svd.cu:123-131 and :159-198, in the same order)
                float cj[ROWS], ck[ROWS];
#pragma unroll
                for (int i = 0; i < ROWS; ++i) { cj[i] = A[i * COLS + j]; ck[i] = A[i * COLS + k]; }
                float p = 0.f, sa = 0.f, qa = 1.f, sb = 0.f, qb = 1.f;
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    const float xj = cj[i], xk = ck[i];
                    p += xj * xk;
                    if (xj != 0.f) {
                        const float ax = fabsf(xj);
                        if (sa < ax) { qa = 1.f + qa * (sa / ax) * (sa / ax); sa = ax; }
                        else qa += (ax / sa) * (ax / sa);
                    }
                    if (xk != 0.f) {
                        const float ax = fabsf(xk);
                        if (sb < ax) { qb = 1.f + qb * (sb / ax) * (sb / ax); sb = ax; }
                        else qb += (ax / sb) * (ax / sb);
                    }
                }
                p *= 2.0f;
                const float a = sa * sqrtf(qa), b = sb * sqrtf(qb);
                const float q = a * a - b * b;
                const float v = hyp(p, q);
                const float ea = err[j], eb = err[k];
                const bool sorted = a >= b;
                const bool orthog = fabsf(p) <= tol * (a * b);
                if (sorted && (orthog || a < ea || b < eb)) { --count; continue; }
                float c, s;
                if (v == 0.f || !sorted) { c = 0.f; s = 1.f; }
                else {
                    c = (float)sqrt((double)(v + q) / (2.0 * (double)v));
                    s = (float)((double)p / (2.0 * (double)v * (double)c));
                }
#pragma unroll
                for (int i = 0; i < ROWS; ++i) {
                    const float Aik = ck[i], Aij = cj[i];
                    A[i * COLS + j] = Aij * c + Aik * s;
                    A[i * COLS + k] = -Aij * s + Aik * c;
                }
                err[j] = fabsf(c) * ea + fabsf(s) * eb;
                err[k] = fabsf(s) * ea + fabsf(c) * eb;
#pragma unroll
                for (int i = 0; i < COLS; ++i) {
                    const float Qij = Q[i * COLS + j], Qik = Q[i * COLS + k];
                    Q[i * COLS + j] = Qij * c + Qik * s;
                    Q[i * COLS + k] = -Qij * s + Qik * c;
                }
            }
        ++sweep;
    }
}

// inv(dst_transform) * H * src_transform, expanded (ransac.cu:201-212, :424-434)
__device__ void denormalise(const float* H, float s1, float s2, float tx1, float ty1, float tx2, float ty2, float* R)
{
    R[0] = s1 * tx2 * H[6] + s1 * H[0] / s2;
    R[1] = s1 * tx2 * H[7] + s1 * H[1] / s2;
    R[2] = tx2 * (H[8] - s1 * ty1 * H[7] - s1 * tx1 * H[6]) + (H[2] - s1 * ty1 * H[1] - s1 * tx1 * H[0]) / s2;
    R[3] = s1 * ty2 * H[6] + s1 * H[3] / s2;
    R[4] = s1 * ty2 * H[7] + s1 * H[4] / s2;
    R[5] = ty2 * (H[8] - s1 * ty1 * H[7] - s1 * tx1 * H[6]) + (H[5] - s1 * ty1 * H[4] - s1 * tx1 * H[3]) / s2;
    R[6] = s1 * H[6];
    R[7] = s1 * H[7];
    R[8] = H[8] - s1 * ty1 * H[7] - s1 * tx1 * H[6];
}

// centroid, mean squared distance, sqrt(2)/rms scale of M points (ransac.cu:100-118, :326-341)
template <int M>
__device__ void normaliser(const float2* p, float& mx, float& my, float& scale)
{
    float sx = p[0].x, sy = p[0].y;
#pragma unroll
    for (int i = 1; i < M; ++i) { sx += p[i].x; sy += p[i].y; }
    mx = sx * (1.0f / M); my = sy * (1.0f / M);
    float var = 0.f;
#pragma unroll
    for (int i = 0; i < M; ++i) var += (p[i].x - mx) * (p[i].x - mx) + (p[i].y - my) * (p[i].y - my);
    if (M == 2) var = (float)((double)var * 0.5);       // ransac.cu:336-337 multiply by a double literal
    else var *= 0.25f;
    scale = sqrtf(2.0f) / sqrtf(var);
}

// 4-point homography, ransac.cu:84-214: nine DLT rows (the two of every point + the third of point 3)
__device__ void homography4(const float2* src, const float2* dst, float* R, SMat X, SMat V, SMat err)
{
    float smx, smy, s1, dmx, dmy, s2;
    normaliser<4>(src, smx, smy, s1);
    normaliser<4>(dst, dmx, dmy, s2);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float a = (src[i].x - smx) * s1, b = (src[i].y - smy) * s1;
        const float u = (dst[i].x - dmx) * s2, w = (dst[i].y - dmy) * s2;
        const float r1[9] = {0.f, 0.f, 0.f, -a, -b, -1.f, w * a, w * b, w};
        const float r2[9] = {a, b, 1.f, 0.f, 0.f, 0.f, -u * a, -u * b, -u};
#pragma unroll
        for (int e = 0; e < 9; ++e) { X[18 * i + e] = r1[e]; X[18 * i + 9 + e] = r2[e]; }
        if (i == 3) {
            const float r3[9] = {-w * a, -w * b, -w, u * a, u * b, u, 0.f, 0.f, 0.f};
#pragma unroll
            for (int e = 0; e < 9; ++e) X[72 + e] = r3[e];
        }
    }
    jacobi_right_vectors<9, 9>(X, V, err);
    float H[9];
    const float div = V[80];
#pragma unroll
    for (int i = 0; i < 8; ++i) H[i] = V[i * 9 + 8] / div;
    H[8] = 1.f;
    denormalise(H, s1, s2, smx, smy, dmx, dmy, R);
}

// 2-point similarity, ransac.cu:320-435: 4 x 5 system in (a, tx, b, ty, 1)
__device__ void similarity2(const float2* src, const float2* dst, float* R, SMat X, SMat V, SMat err)
{
    float smx, smy, s1, dmx, dmy, s2;
    normaliser<2>(src, smx, smy, s1);
    normaliser<2>(dst, dmx, dmy, s2);
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const float a = (src[i].x - smx) * s1, b = (src[i].y - smy) * s1;
        const float u = (dst[i].x - dmx) * s2, w = (dst[i].y - dmy) * s2;
        const float r1[5] = {a, 1.f, -b, 0.f, u};
        const float r2[5] = {b, 0.f, a, 1.f, w};
#pragma unroll
        for (int e = 0; e < 5; ++e) { X[10 * i + e] = r1[e]; X[10 * i + 5 + e] = r2[e]; }
    }
    jacobi_right_vectors<4, 5>(X, V, err);
    const float div = V[24];
    const float a0 = -V[4] / div, a1 = -V[9] / div, b0 = -V[14] / div, b1 = -V[19] / div;
    const float H[9] = {a0, -b0, a1, b0, a0, b1, 0.f, 0.f, 1.f};
    denormalise(H, s1, s2, smx, smy, dmx, dmy, R);
}

// ---- kernels -----------------------------------------------------------------------------------
// establish_correspondences (ransac.cu:29-48)
__global__ void align_kernel(const float* __restrict__ src_x, const float* __restrict__ src_y,
                             const float* __restrict__ dst_x, const float* __restrict__ dst_y,
                             float* __restrict__ c_src_x, float* __restrict__ c_src_y,
                             float* __restrict__ c_dst_x, float* __restrict__ c_dst_y,
                             const int* __restrict__ matches, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int m = matches[i];
    const bool ok = m != -1;
    c_src_x[i] = ok ? src_x[i] : -1.f;
    c_src_y[i] = ok ? src_y[i] : -1.f;
    c_dst_x[i] = ok ? dst_x[m] : -1.f;
    c_dst_y[i] = ok ? dst_y[m] : -1.f;
}

// align_points for the links of a SIFT batch in the span layout (nm_span_links): link l = (frame t, frame t + d), sizes
// on the device; span 1 = the consecutive pairs
__global__ void align_pairs_kernel(const float* __restrict__ x, const float* __restrict__ y, const int* __restrict__ matches,
                                   const int* __restrict__ counts, int n_frames, int capacity, float* __restrict__ c_src_x,
                                   float* __restrict__ c_src_y, float* __restrict__ c_dst_x, float* __restrict__ c_dst_y)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x, l = blockIdx.y;
    if (i >= capacity) return;
    int t, d;
    nm_link_decode(l, n_frames, t, d);
    const long long o = (long long)l * capacity + i, a = (long long)t * capacity + i;
    const int nA = min(counts[t], capacity), nB = min(counts[t + d], capacity);
    const int m = i < nA ? matches[o] : -1;
    const bool ok = m >= 0 && m < nB;
    c_src_x[o] = ok ? x[a] : -1.f;
    c_src_y[o] = ok ? y[a] : -1.f;
    c_dst_x[o] = ok ? x[a + (long long)d * capacity - i + m] : -1.f;
    c_dst_y[o] = ok ? y[a + (long long)d * capacity - i + m] : -1.f;
}

// ---- batched estimator: every kernel indexes a PAIR of frames by a grid dimension ------------------------
// Pair p reads its correspondences at (sx, sy, dx, dy) + p * stride, n(p) = counts ? min(counts[p], max_pts) :
// max_pts of them; per-pair workspace slices: valid[p * max_pts], state[p * 4], rand[p * draws], H[p * it * 9],
// inliers / skip [p * it].  A single estimate is the batch of one.
struct Pairs {
    const float *sx, *sy, *dx, *dy;
    long long stride;
    const int* counts;
    int max_pts;
};
__device__ __forceinline__ int pair_n(const Pairs& P, int p)
{
    if (P.counts == nullptr) return P.max_pts;
    const int c = P.counts[p];
    return c < 0 ? 0 : (c < P.max_pts ? c : P.max_pts);
}

// Ordered list of the indices with src_x >= 0 (the host loop of ransac.cu:533-538); one CTA per pair.
// state[p * 4] = number of valid correspondences.
__global__ void __launch_bounds__(1024) valid_list_kernel(const Pairs P, int* __restrict__ list_all, int* __restrict__ state_all)
{
    __shared__ int warp_tot[32];
    __shared__ int base;
    const int p = blockIdx.x, n = pair_n(P, p);
    const float* __restrict__ src_x = P.sx + (long long)p * P.stride;
    int* __restrict__ list = list_all + (long long)p * P.max_pts;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) base = 0;
    __syncthreads();
    for (int start = 0; start < n; start += 1024) {
        const int i = start + tid;
        const bool ok = i < n && src_x[i] >= 0.f;
        const unsigned m = __ballot_sync(0xffffffffu, ok);
        if (lane == 0) warp_tot[wid] = __popc(m);
        __syncthreads();
        int off = base;
        for (int w = 0; w < wid; ++w) off += warp_tot[w];
        if (ok) list[off + __popc(m & ((1u << lane) - 1))] = i;
        __syncthreads();
        if (tid == 0) {
            int t = 0;
            for (int w = 0; w < 32; ++w) t += warp_tot[w];
            base += t;
        }
        __syncthreads();
    }
    if (tid == 0) state_all[p * 4] = base;
}

__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

// rand_list[d] = valid[u(seed + p, d) scaled to [0, n_valid)], d < draws (the host loop of ransac.cu:551-555)
__global__ void draw_kernel(const int* __restrict__ valid_all, const int* __restrict__ state_all, int max_pts, int min_pts,
                            unsigned long long seed, int draws, int* __restrict__ rand_all)
{
    const int d = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (d >= draws) return;
    int* rand_list = rand_all + (long long)p * draws;
    const int nv = state_all[p * 4];
    if (nv < min_pts) { rand_list[d] = 0; return; }
    const unsigned r = (unsigned)(splitmix64((seed + (unsigned long long)p) ^ (0xD1B54A32D192ED03ull * (unsigned long long)(d + 1))) >> 32);
    rand_list[d] = valid_all[(long long)p * max_pts + (int)(((unsigned long long)r * (unsigned)nv) >> 32)];
}

// One thread per (pair, iteration): the hypothesis (translation_kernel / similarity_transformation_kernel /
// homography_kernel, ransac.cu:437-520, without their scoring loop).  skip = 1 for an iteration with a
// repeated index: H stays 0 and it scores 0, as in the reference (zero-filled buffers, early return).
// CTAs of kHypThreads = 32: a hypothesis is one long dependent chain (5-9 Jacobi sweeps of 36 rotations), so
// the hypotheses are spread over as many SMs as possible instead of packed 128 or 256 to a CTA.
template <int KIND>
__global__ void __launch_bounds__(kHypThreads) hypothesis_kernel(const Pairs P, const int* __restrict__ rand_all, int iterations,
                                                                 const int* __restrict__ state_all, int min_pts,
                                                                 float* __restrict__ H_all, int* __restrict__ inliers,
                                                                 unsigned char* __restrict__ skip)
{
    constexpr int M = KIND == 0 ? 1 : KIND == 1 ? 2 : 4;
    __shared__ float ws[KIND == 0 ? 1 : (81 + 81 + 9) * kHypThreads];
    const SMat X{ws + threadIdx.x}, V{ws + 81 * kHypThreads + threadIdx.x}, err{ws + 162 * kHypThreads + threadIdx.x};
    const int it = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (it >= iterations) return;
    const long long off = (long long)p * P.stride;
    const float* __restrict__ sx = P.sx + off;
    const float* __restrict__ sy = P.sy + off;
    const float* __restrict__ dx = P.dx + off;
    const float* __restrict__ dy = P.dy + off;
    const int* __restrict__ rand_list = rand_all + (long long)p * iterations * M;
    float H[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) H[i] = 0.f;
    int r[M];
#pragma unroll
    for (int i = 0; i < M; ++i) r[i] = rand_list[it * M + i];
    bool dup = state_all != nullptr && state_all[p * 4] < min_pts;      // not enough correspondences: nothing is estimated
    const int n = pair_n(P, p);
#pragma unroll
    for (int a = 0; a < M; ++a) {
        dup |= (unsigned)r[a] >= (unsigned)n;                           // a caller's list with an index outside the arrays
#pragma unroll
        for (int b = a + 1; b < M; ++b) dup |= r[a] == r[b];
    }
    if (!dup) {
        float2 src[M], dst[M];
#pragma unroll
        for (int i = 0; i < M; ++i) {
            src[i] = make_float2(sx[r[i]], sy[r[i]]);
            dst[i] = make_float2(dx[r[i]], dy[r[i]]);
        }
        if (KIND == 0) {                                     // compute_translation, ransac.cu:304-310
            H[0] = H[4] = H[8] = 1.f;
            H[2] = dst[0].x - src[0].x;
            H[5] = dst[0].y - src[0].y;
        } else if (KIND == 1) similarity2(src, dst, H, X, V, err);
        else homography4(src, dst, H, X, V, err);
    }
    const long long o = (long long)p * iterations + it;
#pragma unroll
    for (int i = 0; i < 9; ++i) H_all[o * 9 + i] = H[i];
    inliers[o] = 0;
    skip[o] = dup ? 1 : 0;
}

// eval_transformation (ransac.cu:61-82) for 128 hypotheses x one block of up to 256 correspondences of one pair
// (two IEEE divisions per evaluation make the loop long: short blocks give the grid enough CTAs to fill the SMs).
constexpr int kScoreThreads = 128, kScorePts = 256;
__global__ void __launch_bounds__(kScoreThreads) score_kernel(const Pairs P, const float* __restrict__ H_all,
                                                              const unsigned char* __restrict__ skip, int iterations, float thr,
                                                              int* __restrict__ inliers)
{
    __shared__ float4 pts[kScorePts];
    const int p = blockIdx.z, n = pair_n(P, p);
    const int p0 = blockIdx.y * kScorePts, np = min(kScorePts, n - p0);
    if (np <= 0) return;
    const long long off = (long long)p * P.stride + p0;
    for (int i = threadIdx.x; i < np; i += kScoreThreads) pts[i] = make_float4(P.sx[off + i], P.sy[off + i], P.dx[off + i], P.dy[off + i]);
    __syncthreads();
    const int it = blockIdx.x * kScoreThreads + threadIdx.x;
    const long long o = (long long)p * iterations + it;
    if (it >= iterations || skip[o]) return;
    float H[9];
#pragma unroll
    for (int i = 0; i < 9; ++i) H[i] = H_all[o * 9 + i];
    int cnt = 0;
    for (int i = 0; i < np; ++i) {
        const float4 q = pts[i];
        if (q.x >= 0.f) {
            float x = H[0] * q.x + H[1] * q.y + H[2];
            float y = H[3] * q.x + H[4] * q.y + H[5];
            const float z = H[6] * q.x + H[7] * q.y + H[8];
            x /= z;
            y /= z;
            const float d2 = (q.z - x) * (q.z - x) + (q.w - y) * (q.w - y);
            if (d2 < thr) ++cnt;
        }
    }
    if (cnt) atomicAdd(inliers + o, cnt);
}

// thrust::max_element (first maximum, ransac.cu:566-570) + the 9-float copy; one CTA per pair.
// status[p*3 + 0] = 1 when a model was written, 0 when there were too few correspondences (the reference returns
// false and leaves `homography` untouched); [1] = inlier count of the chosen hypothesis, [2] = its index.
__global__ void __launch_bounds__(256) select_kernel(const int* __restrict__ inliers_all, const float* __restrict__ H_all, int iterations,
                                                     const int* __restrict__ state_all, int min_pts, float* __restrict__ H_out_all,
                                                     int* __restrict__ status_all)
{
    __shared__ long long best[256];
    const int tid = threadIdx.x, p = blockIdx.x;
    int* status = status_all + p * 3;
    if (state_all[p * 4] < min_pts) {
        if (tid == 0) { status[0] = 0; status[1] = 0; status[2] = -1; }
        return;
    }
    const int* inliers = inliers_all + (long long)p * iterations;
    // key = count in the high word, ~index in the low word: a larger key is a larger count, then a smaller index
    long long key = -1;
    for (int i = tid; i < iterations; i += 256) {
        const long long k = ((long long)inliers[i] << 32) | (unsigned)(0x7fffffff - i);
        key = k > key ? k : key;
    }
    best[tid] = key;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if (tid < s && best[tid + s] > best[tid]) best[tid] = best[tid + s];
        __syncthreads();
    }
    const int idx = 0x7fffffff - (int)(best[0] & 0xffffffffll);
    if (tid < 9) H_out_all[p * 9 + tid] = H_all[((long long)p * iterations + idx) * 9 + tid];
    if (tid == 0) { status[0] = 1; status[1] = (int)(best[0] >> 32); status[2] = idx; }
}

// score_kernel's inlier rule, expression for expression: q = (src_x, src_y, dst_x, dst_y) is an inlier of H when
// src_x >= 0 and the squared forward transfer error is < thr.  The mask of a RANSAC model therefore has exactly as many
// bits set as the model's score (tests/test_gpu_ransac_refine.py).  score_kernel keeps its own copy of the loop body:
// calling any helper there, this one included, changes how its loop is unrolled.
__device__ __forceinline__ bool transfer_inlier(const float* H, const float4 q, float thr)
{
    if (!(q.x >= 0.f)) return false;
    float x = H[0] * q.x + H[1] * q.y + H[2];
    float y = H[3] * q.x + H[4] * q.y + H[5];
    const float z = H[6] * q.x + H[7] * q.y + H[8];
    x /= z;
    y /= z;
    const float d2 = (q.z - x) * (q.z - x) + (q.w - y) * (q.w - y);
    return d2 < thr;
}

// ---- refit of a model on its inlier set (no reference counterpart) ------------------------------------------------
// One CTA per pair.  An inlier set is never stored: every pass over it applies transfer_inlier with the set's fp32
// model to the pair's correspondences (read from L2 after the first pass), so no workspace is needed and sets of any
// size take the same path.  Sums are fp64: each thread adds its correspondences in index order, each warp folds its
// lanes in a fixed butterfly, then the warps are added in order -- bit-reproducible, and pair p depends on nothing
// but its own inputs.
constexpr int kRefineThreads = 256, kRefineWarps = kRefineThreads / 32, kRefineSums = 29;
constexpr int kLmIterations = 20, kJacobiSweeps = 30;

struct RefineShared {
    float H[2][9];                              // [0] model of the current inlier set, [1] the refit
    double red[kRefineWarps][kRefineSums];      // per-warp partial sums
    double tot[kRefineSums];                    // block sums
    double A[81], V[81];                        // DLT normal matrix (eigenvalues on its diagonal after Jacobi), eigenvectors
    double J[64], g[8], L[64];                  // LM normal equations J^T J, J^T r, Cholesky factor
    double prm[2][8];                           // LM point and trial point (normalised homography, h8 = 1)
    int ok;
};

template <int K>
__device__ void block_sum(double (&v)[K], RefineShared& S)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < K; ++k) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
        if (lane == 0) S.red[wid][k] = v[k];
    }
    __syncthreads();
    for (int k = threadIdx.x; k < K; k += kRefineThreads) {
        double s = S.red[0][k];
        for (int w = 1; w < kRefineWarps; ++w) s += S.red[w][k];
        S.tot[k] = s;
    }
    __syncthreads();
}

// f(q) for every correspondence q of pair p that is an inlier of the fp32 model Hsh
template <class F>
__device__ __forceinline__ void for_each_inlier(const Pairs& P, int p, int n, const float* Hsh, float thr, F f)
{
    float H[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) H[k] = Hsh[k];
    const long long off = (long long)p * P.stride;
    for (int i = threadIdx.x; i < n; i += kRefineThreads) {
        const float4 q = make_float4(P.sx[off + i], P.sy[off + i], P.dx[off + i], P.dy[off + i]);
        if (transfer_inlier(H, q, thr)) f(q);
    }
}

// Hartley normalisation of both point sets: src (x - mx) * s, dst likewise, RMS distance from the centroid sqrt(2)
struct Norm {
    double smx, smy, s1, dmx, dmy, s2;
    __device__ void apply(const float4 q, double& a, double& b, double& u, double& v) const
    {
        a = ((double)q.x - smx) * s1;
        b = ((double)q.y - smy) * s1;
        u = ((double)q.z - dmx) * s2;
        v = ((double)q.w - dmy) * s2;
    }
};

// Solves A x = b for a symmetric positive definite N x N matrix whose lower triangle is in L (overwritten by the
// factor).  False when a pivot is not positive or the solution is not finite.
template <int N>
__device__ bool cholesky_solve(double* L, const double* b, double* x)
{
    for (int j = 0; j < N; ++j) {
        double d = L[j * N + j];
        for (int k = 0; k < j; ++k) d -= L[j * N + k] * L[j * N + k];
        if (!(d > 0.0)) return false;
        d = sqrt(d);
        L[j * N + j] = d;
        for (int i = j + 1; i < N; ++i) {
            double s = L[i * N + j];
            for (int k = 0; k < j; ++k) s -= L[i * N + k] * L[j * N + k];
            L[i * N + j] = s / d;
        }
    }
    for (int i = 0; i < N; ++i) {
        double s = b[i];
        for (int k = 0; k < i; ++k) s -= L[i * N + k] * x[k];
        x[i] = s / L[i * N + i];
    }
    bool ok = true;
    for (int i = N - 1; i >= 0; --i) {
        double s = x[i];
        for (int k = i + 1; k < N; ++k) s -= L[k * N + i] * x[k];
        x[i] = s / L[i * N + i];
        ok &= isfinite(x[i]);
    }
    return ok;
}

// Cyclic Jacobi on the symmetric 9 x 9 matrix A (eigenvalues on its diagonal afterwards), eigenvectors to the columns
// of V.  Called by warp 0: every lane decides the same rotations, lane k < 9 rotates row and column k.
__device__ void jacobi_eigen9(double* A, double* V)
{
    const int k = threadIdx.x;
    for (int i = k; i < 81; i += 32) V[i] = i % 10 == 0 ? 1.0 : 0.0;
    __syncwarp();
    for (int sweep = 0; sweep < kJacobiSweeps; ++sweep) {
        bool rotated = false;
        for (int p = 0; p < 8; ++p)
            for (int q = p + 1; q < 9; ++q) {
                const double apq = A[p * 9 + q], app = A[p * 9 + p], aqq = A[q * 9 + q];
                __syncwarp();
                if (!(fabs(apq) > 1e-18 * sqrt(fabs(app * aqq)))) continue;
                const double theta = (aqq - app) / (2.0 * apq), at = fabs(theta);
                const double t = at > 1e100 ? 0.5 / theta : (theta >= 0.0 ? 1.0 : -1.0) / (at + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                if (k < 9) {
                    const double akp = A[k * 9 + p], akq = A[k * 9 + q];
                    A[k * 9 + p] = c * akp - s * akq;
                    A[k * 9 + q] = s * akp + c * akq;
                }
                __syncwarp();
                if (k < 9) {
                    const double apk = A[p * 9 + k], aqk = A[q * 9 + k];
                    A[p * 9 + k] = c * apk - s * aqk;
                    A[q * 9 + k] = s * apk + c * aqk;
                    const double vkp = V[k * 9 + p], vkq = V[k * 9 + q];
                    V[k * 9 + p] = c * vkp - s * vkq;
                    V[k * 9 + q] = s * vkp + c * vkq;
                }
                __syncwarp();
                if (k == 0) A[p * 9 + q] = A[q * 9 + p] = 0.0;
                __syncwarp();
                rotated = true;
            }
        if (!rotated) break;
    }
}

// out = fp32 of Td^-1 . Hn . Ts divided by its [8]; false when not finite
__device__ bool denormalise_store(const double* Hn, const Norm& nm, float* out)
{
    double T[9], R[9];
    for (int r = 0; r < 3; ++r) {
        T[r * 3 + 0] = Hn[r * 3 + 0] * nm.s1;
        T[r * 3 + 1] = Hn[r * 3 + 1] * nm.s1;
        T[r * 3 + 2] = Hn[r * 3 + 2] - Hn[r * 3 + 0] * nm.s1 * nm.smx - Hn[r * 3 + 1] * nm.s1 * nm.smy;
    }
    for (int c = 0; c < 3; ++c) {
        R[c] = T[c] / nm.s2 + nm.dmx * T[6 + c];
        R[3 + c] = T[3 + c] / nm.s2 + nm.dmy * T[6 + c];
        R[6 + c] = T[6 + c];
    }
    bool ok = true;
    for (int e = 0; e < 9; ++e) {
        out[e] = (float)(R[e] / R[8]);
        ok &= isfinite(out[e]);
    }
    return ok;
}

// sum of squared forward transfer errors in normalised coordinates at the normalised homography h (h8 = 1)
__device__ double lm_cost(const Pairs& P, int p, int n, float thr, const Norm& nm, const double* hs, RefineShared& S)
{
    double h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) h[e] = hs[e];
    double v[1] = {0.0};
    for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
        double a, b, u, w;
        nm.apply(q, a, b, u, w);
        const double iw = 1.0 / (h[6] * a + h[7] * b + 1.0);
        const double rx = (h[0] * a + h[1] * b + h[2]) * iw - u, ry = (h[3] * a + h[4] * b + h[5]) * iw - w;
        v[0] += rx * rx + ry * ry;
    });
    block_sum(v, S);
    return S.tot[0];
}

// J^T J and J^T r of the transfer error at h: with g = (a, b, 1) / w, c = (a, b) / w and the mapped point (X, Y), the
// Jacobian rows are [g, 0, -X c] and [0, g, -Y c], so 29 sums make up the 8 x 8 system (written by thread 0).
__device__ void lm_normal(const Pairs& P, int p, int n, float thr, const Norm& nm, const double* hs, RefineShared& S)
{
    double h[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) h[e] = hs[e];
    double v[kRefineSums];
#pragma unroll
    for (int e = 0; e < kRefineSums; ++e) v[e] = 0.0;
    for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
        double a, b, u, w;
        nm.apply(q, a, b, u, w);
        const double iw = 1.0 / (h[6] * a + h[7] * b + 1.0);
        const double X = (h[0] * a + h[1] * b + h[2]) * iw, Y = (h[3] * a + h[4] * b + h[5]) * iw;
        const double rx = X - u, ry = Y - w;
        const double g[3] = {a * iw, b * iw, iw};
        v[0] += g[0] * g[0]; v[1] += g[0] * g[1]; v[2] += g[0] * g[2];
        v[3] += g[1] * g[1]; v[4] += g[1] * g[2]; v[5] += g[2] * g[2];
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const double xg = X * g[i], yg = Y * g[i];
            v[6 + 2 * i] += xg * g[0]; v[7 + 2 * i] += xg * g[1];
            v[12 + 2 * i] += yg * g[0]; v[13 + 2 * i] += yg * g[1];
            v[21 + i] += rx * g[i];
            v[24 + i] += ry * g[i];
        }
        const double q2 = X * X + Y * Y, e = X * rx + Y * ry;
        v[18] += q2 * g[0] * g[0]; v[19] += q2 * g[0] * g[1]; v[20] += q2 * g[1] * g[1];
        v[27] -= e * g[0]; v[28] -= e * g[1];
    });
    block_sum(v, S);
    if (threadIdx.x == 0) {
        const double* t = S.tot;
        const int s3[9] = {0, 1, 2, 1, 3, 4, 2, 4, 5};
        for (int e = 0; e < 64; ++e) S.J[e] = 0.0;
        for (int i = 0; i < 3; ++i) {
            for (int j = 0; j < 3; ++j) S.J[i * 8 + j] = S.J[(3 + i) * 8 + 3 + j] = t[s3[i * 3 + j]];
            for (int j = 0; j < 2; ++j) {
                S.J[i * 8 + 6 + j] = S.J[(6 + j) * 8 + i] = -t[6 + 2 * i + j];
                S.J[(3 + i) * 8 + 6 + j] = S.J[(6 + j) * 8 + 3 + i] = -t[12 + 2 * i + j];
            }
        }
        S.J[6 * 8 + 6] = t[18];
        S.J[6 * 8 + 7] = S.J[7 * 8 + 6] = t[19];
        S.J[7 * 8 + 7] = t[20];
        for (int e = 0; e < 8; ++e) S.g[e] = t[21 + e];
    }
}

// Least-squares refit on the inlier set of S.H[0] (cnt correspondences) into S.H[1].  False when the fit is degenerate
// or its fp32 result is not finite; S.H[1] is then not used.
template <int KIND>
__device__ bool refit(const Pairs& P, int p, int n, float thr, int cnt, RefineShared& S)
{
    const int tid = threadIdx.x;
    const double N = (double)cnt;
    if constexpr (KIND == 0) {                                   // the mean displacement
        double v[2] = {0.0, 0.0};
        for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
            v[0] += (double)q.z - (double)q.x;
            v[1] += (double)q.w - (double)q.y;
        });
        block_sum(v, S);
        if (tid == 0) {
            const float H[9] = {1.f, 0.f, (float)(S.tot[0] / N), 0.f, 1.f, (float)(S.tot[1] / N), 0.f, 0.f, 1.f};
            for (int e = 0; e < 9; ++e) S.H[1][e] = H[e];
            S.ok = isfinite(H[2]) && isfinite(H[5]);
        }
        __syncthreads();
        return S.ok;
    } else {
    Norm nm;
    {
        double v[4] = {0.0, 0.0, 0.0, 0.0};
        for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) { v[0] += q.x; v[1] += q.y; v[2] += q.z; v[3] += q.w; });
        block_sum(v, S);
        nm.smx = S.tot[0] / N; nm.smy = S.tot[1] / N; nm.dmx = S.tot[2] / N; nm.dmy = S.tot[3] / N;
        nm.s1 = nm.s2 = 1.0;
        double r[2] = {0.0, 0.0};
        for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
            double a, b, u, w;
            nm.apply(q, a, b, u, w);
            r[0] += a * a + b * b;
            r[1] += u * u + w * w;
        });
        block_sum(r, S);
        nm.s1 = sqrt(2.0) / sqrt(S.tot[0] / N);
        nm.s2 = sqrt(2.0) / sqrt(S.tot[1] / N);
    }
    if constexpr (KIND == 1) {
        // u = a' x - b' y + tx, v = b' x + a' y + ty is linear in (a', b', tx, ty): 4 x 4 normal equations
        double v[7];
#pragma unroll
        for (int e = 0; e < 7; ++e) v[e] = 0.0;
        for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
            double x, y, u, w;
            nm.apply(q, x, y, u, w);
            v[0] += x * x + y * y; v[1] += x; v[2] += y;
            v[3] += x * u + y * w; v[4] += x * w - y * u; v[5] += u; v[6] += w;
        });
        block_sum(v, S);
        if (tid == 0) {
            const double* t = S.tot;
            const double A[16] = {t[0], 0.0, t[1], t[2], 0.0, t[0], -t[2], t[1], t[1], -t[2], N, 0.0, t[2], t[1], 0.0, N};
            for (int e = 0; e < 16; ++e) S.L[e] = A[e];
            double x[4];
            bool ok = cholesky_solve<4>(S.L, t + 3, x);
            const double Hn[9] = {x[0], -x[1], x[2], x[1], x[0], x[3], 0.0, 0.0, 1.0};
            S.ok = ok && denormalise_store(Hn, nm, S.H[1]);
        }
        __syncthreads();
        return S.ok;
    } else {
    // homography: normalised DLT, the two rows per point of homography4, M = sum r^T r from 24 sums of t t^T, t = (a, b, 1)
    {
        double v[24];
#pragma unroll
        for (int e = 0; e < 24; ++e) v[e] = 0.0;
        for_each_inlier(P, p, n, S.H[0], thr, [&](const float4 q) {
            double a, b, u, w;
            nm.apply(q, a, b, u, w);
            const double tt[6] = {a * a, a * b, a, b * b, b, 1.0};
            const double q2 = u * u + w * w;
#pragma unroll
            for (int e = 0; e < 6; ++e) {
                v[e] += tt[e];
                v[6 + e] += u * tt[e];
                v[12 + e] += w * tt[e];
                v[18 + e] += q2 * tt[e];
            }
        });
        block_sum(v, S);
        if (tid < 81) {
            const int i = tid / 9, j = tid % 9, bi = i / 3, bj = j / 3;
            const int s3[9] = {0, 1, 2, 1, 3, 4, 2, 4, 5};
            const double m = S.tot[s3[(i % 3) * 3 + j % 3]], mu = S.tot[6 + s3[(i % 3) * 3 + j % 3]];
            const double mw = S.tot[12 + s3[(i % 3) * 3 + j % 3]], mq = S.tot[18 + s3[(i % 3) * 3 + j % 3]];
            double x = 0.0;                                    // blocks of M: [S0 0 -Su; 0 S0 -Sw; -Su -Sw Sq]
            if (bi == bj) x = bi == 2 ? mq : m;
            else if (bi == 2 || bj == 2) x = (bi == 0 || bj == 0) ? -mu : -mw;
            S.A[tid] = x;
        }
        __syncthreads();
        if (tid < 32) {
            jacobi_eigen9(S.A, S.V);
            if (tid == 0) {
                int lo = 0;
                double hi = S.A[0];
                for (int e = 1; e < 9; ++e) {
                    if (S.A[e * 10] < S.A[lo * 10]) lo = e;
                    hi = fmax(hi, S.A[e * 10]);
                }
                double second = INFINITY;
                for (int e = 0; e < 9; ++e)
                    if (e != lo) second = fmin(second, S.A[e * 10]);
                const double h8 = S.V[8 * 9 + lo];
                // a null space of more than one dimension (collinear points, ...) or a model at infinity
                S.ok = second > 1e-12 * hi && fabs(h8) > 1e-12;
                for (int e = 0; e < 8; ++e) S.prm[0][e] = S.V[e * 9 + lo] / h8;
            }
        }
        __syncthreads();
        if (!S.ok) return false;
    }
    // Levenberg-Marquardt on the transfer error: lambda0 = 1e-3 max diag(J^T J), (J^T J + lambda diag) d = -J^T r,
    // accepted step -> lambda / 10, rejected -> lambda * 10; at most kLmIterations steps, stop when an accepted step
    // gains less than 1e-12 of the cost or when lambda > 1e16.  Every thread keeps the same (cur, cost, lambda).
    int cur = 0;
    double cost = lm_cost(P, p, n, thr, nm, S.prm[0], S);
    lm_normal(P, p, n, thr, nm, S.prm[0], S);
    double lambda = 1e-3 * fmax(fmax(fmax(S.tot[0], S.tot[3]), fmax(S.tot[5], S.tot[18])), S.tot[20]);
    for (int it = 0; it < kLmIterations; ++it) {
        if (tid == 0) {
            for (int e = 0; e < 64; ++e) S.L[e] = S.J[e];
            for (int e = 0; e < 8; ++e) S.L[e * 9] += lambda * S.J[e * 9];
            double d[8], rhs[8];
            for (int e = 0; e < 8; ++e) rhs[e] = -S.g[e];
            S.ok = cholesky_solve<8>(S.L, rhs, d);
            for (int e = 0; e < 8; ++e) S.prm[cur ^ 1][e] = S.prm[cur][e] + d[e];
        }
        __syncthreads();
        const bool solved = S.ok;
        __syncthreads();                                   // S.ok is rewritten by the next step
        const double trial = solved ? lm_cost(P, p, n, thr, nm, S.prm[cur ^ 1], S) : INFINITY;
        if (trial < cost) {
            const bool done = cost - trial < 1e-12 * cost;
            cost = trial;
            cur ^= 1;
            lambda *= 0.1;
            if (done) break;
            lm_normal(P, p, n, thr, nm, S.prm[cur], S);
        } else {
            lambda *= 10.0;
            if (lambda > 1e16) break;
        }
    }
    if (tid == 0) {
        double Hn[9];
        for (int e = 0; e < 8; ++e) Hn[e] = S.prm[cur][e];
        Hn[8] = 1.0;
        S.ok = denormalise_store(Hn, nm, S.H[1]);
    }
    __syncthreads();
    return S.ok;
    }
    }
}

// Pair p: the inlier set S0 of H_in[p]; round r refits on S(r-1), and keeps the refit unless it is degenerate or has
// fewer inliers than S(r-1); it stops early when the set no longer changes.  status_out[p] = {status_in[p][0],
// inliers of the returned model, refits kept}; mask row p = the returned model's inliers.  Pairs without a model
// (status_in[p][0] == 0) get status {0, 0, 0}, a zero mask row, and H_out[p] is not written.
template <int KIND>
__global__ void __launch_bounds__(kRefineThreads, 1) refine_kernel(const Pairs P, float thr, const float* __restrict__ H_in,
                                                                const int* __restrict__ status_in, int rounds, float* H_out,
                                                                int* status_out, unsigned char* __restrict__ mask_all)
{
    constexpr int M = KIND == 0 ? 1 : KIND == 1 ? 2 : 4;     // minimal sample: no refit with no more points than this
    __shared__ RefineShared S;
    const int p = blockIdx.x, n = pair_n(P, p), tid = threadIdx.x;
    const int has = status_in == nullptr ? 1 : status_in[p * 3];
    if (tid < 9) S.H[0][tid] = H_in[p * 9 + tid];
    __syncthreads();                                        // read before written: H_out / status_out may alias the inputs
    unsigned char* mask = mask_all == nullptr ? nullptr : mask_all + (long long)p * P.max_pts;
    if (has == 0) {
        if (mask != nullptr)
            for (int i = tid; i < P.max_pts; i += kRefineThreads) mask[i] = 0;
        if (tid == 0) status_out[p * 3] = status_out[p * 3 + 1] = status_out[p * 3 + 2] = 0;
        return;
    }
    double c[1] = {0.0};
    for_each_inlier(P, p, n, S.H[0], thr, [&](const float4) { c[0] += 1.0; });
    block_sum(c, S);
    int cnt = (int)S.tot[0], kept = 0;
    for (int r = 1; r <= rounds && cnt > M; ++r) {
        if (!refit<KIND>(P, p, n, thr, cnt, S)) break;
        double v[2] = {0.0, 0.0};                           // |S_r| and |S_r xor S_(r-1)|
        {
            float H0[9], H1[9];
#pragma unroll
            for (int e = 0; e < 9; ++e) { H0[e] = S.H[0][e]; H1[e] = S.H[1][e]; }
            const long long off = (long long)p * P.stride;
            for (int i = tid; i < n; i += kRefineThreads) {
                const float4 q = make_float4(P.sx[off + i], P.sy[off + i], P.dx[off + i], P.dy[off + i]);
                const bool a = transfer_inlier(H0, q, thr), b = transfer_inlier(H1, q, thr);
                v[0] += b ? 1.0 : 0.0;
                v[1] += a != b ? 1.0 : 0.0;
            }
        }
        block_sum(v, S);
        const int cnt_r = (int)S.tot[0], changed = (int)S.tot[1];
        if (cnt_r < cnt) break;
        if (tid < 9) S.H[0][tid] = S.H[1][tid];
        __syncthreads();
        cnt = cnt_r;
        kept = r;
        if (changed == 0) break;
    }
    if (mask != nullptr) {
        float H[9];
#pragma unroll
        for (int e = 0; e < 9; ++e) H[e] = S.H[0][e];
        const long long off = (long long)p * P.stride;
        for (int i = tid; i < P.max_pts; i += kRefineThreads)
            mask[i] = i < n && transfer_inlier(H, make_float4(P.sx[off + i], P.sy[off + i], P.dx[off + i], P.dy[off + i]), thr);
    }
    if (tid < 9) H_out[p * 9 + tid] = S.H[0][tid];
    if (tid == 0) {
        status_out[p * 3] = has;
        status_out[p * 3 + 1] = cnt;
        status_out[p * 3 + 2] = kept;
    }
}

// ---- joint adjustment of a window's chain (nm_ransac_adjust_chain_f32; no reference counterpart) -------------------
// Unknowns: G_k, frame k -> frame-0 pixels, k = 1 .. n-1, G_0 = I.  G_k = N^-1 Gn_k N with N = the frame centred and
// scaled by 2 / max(w, h); Gn_k has P = 2 / 4 / 8 parameters (translation / similarity / homography with Gn[8] = 1).
// Residual of correspondence (a, b) on link (t, u = t + d), normalised, by cost:
//   NM_ADJUST_MOSAIC (0):   pi(Gn_t a) - pi(Gn_u b), the disagreement in frame-0 (mosaic) coordinates;
//   NM_ADJUST_TRANSFER (1): pi(Gn_u^-1 Gn_t a) - b, the forward transfer error in frame u, which depends on the
//     relative pose only.  A point with p3 <= 0 or a non-finite residual makes the cost of that point +inf.
// Every sum below is fp64 and is formed in a fixed order, so a window's result is bit-reproducible.
constexpr int kAdjMaxFrames = 1024, kAdjMaxSpan = 8;
constexpr int kAdjSlices = 4;               // CTAs per link in the normal-equation build
constexpr int kAdjThreads = 128;            // threads of a build CTA = correspondences staged per pass
constexpr int kAdjSolveThreads = 256;

template <int KIND> struct AdjFam {
    static constexpr int P = KIND == 0 ? 2 : KIND == 1 ? 4 : 8;
    static constexpr int M = KIND == 0 ? 1 : KIND == 1 ? 2 : 4;       // mask points a link needs
    static constexpr int E = 3 * P * P + 2 * P + 1;                     // J^T J blocks (t,t), (u,u), (t,u), J^T r of t, u, cost
    static constexpr int W = 2 + 4 * P;                                 // staged per point: r, dpi_t (2 x P), dpi_u (2 x P)
};

struct AdjState {
    double lambda, cost, cost0;             // lambda < 0: not initialised yet
    int first, done, accepted;
    int nonfinite;                          // set by a transfer-cost build: a point at x_eval has p3 <= 0 or a non-finite residual
};

struct AdjGeom {
    double cx, cy, s;                       // normalised point = (p - c) * s
    __device__ double2 norm(float x, float y) const { return make_double2(((double)x - cx) * s, ((double)y - cy) * s); }
};

__device__ __forceinline__ int adj_link(int t, int d, int n) { return (d - 1) * n - (d - 1) * d / 2 + t; }

template <int KIND>
__device__ void adj_identity(double* th)
{
    for (int i = 0; i < AdjFam<KIND>::P; ++i) th[i] = 0.0;
    if (KIND == 1) th[0] = 1.0;
    if (KIND == 2) th[0] = th[4] = 1.0;
}

template <int KIND>
__device__ void adj_matrix(const double* th, double* G)
{
    if (KIND == 0) {
        const double g[9] = {1.0, 0.0, th[0], 0.0, 1.0, th[1], 0.0, 0.0, 1.0};
        for (int i = 0; i < 9; ++i) G[i] = g[i];
    } else if (KIND == 1) {
        const double g[9] = {th[0], -th[1], th[2], th[1], th[0], th[3], 0.0, 0.0, 1.0};
        for (int i = 0; i < 9; ++i) G[i] = g[i];
    } else {
        for (int i = 0; i < 8; ++i) G[i] = th[i];
        G[8] = 1.0;
    }
}

// parameters of a normalised matrix, divided by its [8] first
template <int KIND>
__device__ void adj_params(const double* G, double* th)
{
    const double w = G[8];
    if (KIND == 0) { th[0] = G[2] / w; th[1] = G[5] / w; }
    else if (KIND == 1) { th[0] = G[0] / w; th[1] = G[3] / w; th[2] = G[2] / w; th[3] = G[5] / w; }
    else for (int i = 0; i < 8; ++i) th[i] = G[i] / w;
}

// N G N^-1 (to = 1) or N^-1 G N (to = 0)
__device__ void adj_conj(const AdjGeom& g, const double* G, double* R, bool to)
{
    const double s = to ? g.s : 1.0 / g.s, cx = to ? g.cx : -g.cx * g.s, cy = to ? g.cy : -g.cy * g.s;
    // N = [s 0 -s cx; 0 s -s cy; 0 0 1] and N^-1 = [1/s 0 cx; 0 1/s cy; 0 0 1] are both S'(x) = s' (x - c')
    double T[9];                                     // T = G . S'^-1, S'^-1 x = x / s' + c'
    for (int r = 0; r < 3; ++r) {
        T[r * 3 + 0] = G[r * 3 + 0] / s;
        T[r * 3 + 1] = G[r * 3 + 1] / s;
        T[r * 3 + 2] = G[r * 3 + 0] * cx + G[r * 3 + 1] * cy + G[r * 3 + 2];
    }
    for (int c = 0; c < 3; ++c) {                    // R = S' . T, S' x = s' (x - c')
        R[c] = s * (T[c] - cx * T[6 + c]);
        R[3 + c] = s * (T[3 + c] - cy * T[6 + c]);
        R[6 + c] = T[6 + c];
    }
}

// pi(Gn(th) p) and its derivatives du, dv with respect to th
template <int KIND>
__device__ __forceinline__ void adj_project(const double* th, double px, double py, double& U, double& V, double* du, double* dv)
{
    if (KIND == 0) {
        U = px + th[0]; V = py + th[1];
        du[0] = 1.0; du[1] = 0.0; dv[0] = 0.0; dv[1] = 1.0;
    } else if (KIND == 1) {
        U = th[0] * px - th[1] * py + th[2];
        V = th[1] * px + th[0] * py + th[3];
        du[0] = px; du[1] = -py; du[2] = 1.0; du[3] = 0.0;
        dv[0] = py; dv[1] = px; dv[2] = 0.0; dv[3] = 1.0;
    } else {
        const double iw = 1.0 / (th[6] * px + th[7] * py + 1.0);
        U = (th[0] * px + th[1] * py + th[2]) * iw;
        V = (th[3] * px + th[4] * py + th[5]) * iw;
        const double a = px * iw, b = py * iw;
        du[0] = a; du[1] = b; du[2] = iw; du[3] = 0.0; du[4] = 0.0; du[5] = 0.0; du[6] = -U * a; du[7] = -U * b;
        dv[0] = 0.0; dv[1] = 0.0; dv[2] = 0.0; dv[3] = a; dv[4] = b; dv[5] = iw; dv[6] = -V * a; dv[7] = -V * b;
    }
}

// The two rows of A . dGn/dth . v (times sg = +/-1) for A 2 x 3 and a homogeneous v: dGn/dth v is linear in v.
template <int KIND>
__device__ __forceinline__ void adj_dproj(const double* A, const double* v, double sg, double* du, double* dv)
{
    for (int r = 0; r < 2; ++r) {
        const double* a = A + 3 * r;
        double* o = r ? dv : du;
        if (KIND == 0) { o[0] = sg * (a[0] * v[2]); o[1] = sg * (a[1] * v[2]); }
        else if (KIND == 1) {
            o[0] = sg * (a[0] * v[0] + a[1] * v[1]);
            o[1] = sg * (a[1] * v[0] - a[0] * v[1]);
            o[2] = sg * (a[0] * v[2]);
            o[3] = sg * (a[1] * v[2]);
        } else
            for (int i = 0; i < 8; ++i) o[i] = sg * (a[i / 3] * v[i % 3]);
    }
}

// Transfer residual r = pi(p) - b, p = Gn_u^-1 Gn_t a = M a, into q[0..1], and its derivatives into q[2 ..]: with
// A = dpi/dp . Gn_u^-1, dr/dth_t = A (dGn_t/dth_t) a and dr/dth_u = -A (dGn_u/dth_u) p.  False when p3 <= 0 or r is
// not finite.
template <int KIND>
__device__ __forceinline__ bool adj_transfer(const double* Gi, const double* M, double2 a, double2 b, double* q)
{
    constexpr int NP = AdjFam<KIND>::P;
    const double p[3] = {M[0] * a.x + M[1] * a.y + M[2], M[3] * a.x + M[4] * a.y + M[5], M[6] * a.x + M[7] * a.y + M[8]};
    const double iw = 1.0 / p[2], U = p[0] * iw, V = p[1] * iw;
    q[0] = U - b.x;
    q[1] = V - b.y;
    double A[6];                                             // dpi/dp = iw [1 0 -U; 0 1 -V]
    for (int c = 0; c < 3; ++c) {
        A[c] = iw * (Gi[c] - U * Gi[6 + c]);
        A[3 + c] = iw * (Gi[3 + c] - V * Gi[6 + c]);
    }
    const double av[3] = {a.x, a.y, 1.0};
    adj_dproj<KIND>(A, av, 1.0, q + 2, q + 2 + NP);
    adj_dproj<KIND>(A, p, -1.0, q + 2 + 2 * NP, q + 2 + 3 * NP);
    return p[2] > 0.0 && isfinite(q[0]) && isfinite(q[1]);
}

// mask points of every link (i < n(l), mask byte != 0)
__global__ void __launch_bounds__(256) adjust_count_kernel(const Pairs P, const unsigned char* __restrict__ masks, int* __restrict__ npts)
{
    __shared__ int tot;
    const int l = blockIdx.x, n = pair_n(P, l);
    if (threadIdx.x == 0) tot = 0;
    __syncthreads();
    int c = 0;
    for (int i = threadIdx.x; i < n; i += 256) c += masks[(long long)l * P.max_pts + i] != 0;
    atomicAdd(&tot, c);                                      // integer: the total does not depend on the order
    __syncthreads();
    if (threadIdx.x == 0) npts[l] = tot;
}

// One CTA.  Fixed frames j = 1 .. nf-1 (nf = n_fixed): G_j = C_0^-1 C_j of fixed_chain, renormalised; frame j is
// disconnected (G_j = G_(j-1)) when fixed_conn[j] == 0, G_j is not finite, or C_0 is not finite or singular (|det| <=
// 1e-12 max|C_0|^3, nm_chain_step's rule).  Initial poses of the free frames: for k = nf .. n-1 the smallest d <= span
// with frame k-d connected and link (k-d, d) usable (status 1, at least M mask points) gives G_k = G_(k-d) .
// step(H_link) (nm_chain_step, renormalised: place_kernel's chain); without one frame k is disconnected and G_k =
// G_(k-1).  Then the parameters of N G_k N^-1, the links used (both frames connected, the later one free), and the LM
// state.
template <int KIND>
__global__ void __launch_bounds__(256) adjust_init_kernel(int n, int span, AdjGeom geo, const float* __restrict__ H_links,
                                                          const int* __restrict__ link_status, const int* __restrict__ npts,
                                                          int nf, const double* __restrict__ fixed_chain,
                                                          const int* __restrict__ fixed_conn, double* __restrict__ G,
                                                          int* __restrict__ conn, int* __restrict__ used,
                                                          double* __restrict__ x_cur, double* __restrict__ x_eval, AdjState* state)
{
    constexpr int NP = AdjFam<KIND>::P, M = AdjFam<KIND>::M;
    const int tid = threadIdx.x, L = nm_span_links(n, span);
    auto usable = [&](int l) { return link_status[(long long)l * 3] == 1 && npts[l] >= M; };
    if (tid == 0) {
        for (int i = 0; i < 9; ++i) G[i] = (i % 4 == 0) ? 1.0 : 0.0;
        conn[0] = 1;
        if (nf > 1) {
            double c0[9], c0i[9];
            bool base = true;
            for (int i = 0; i < 9; ++i) { c0[i] = fixed_chain[i]; base = base && isfinite(c0[i]); }
            if (base) {
                const double m = nm_max_abs9(c0), det = nm_det3d(c0);
                base = fabs(det) > 1e-12 * m * m * m;
                if (base) nm_inv3d(c0, det, c0i);
            }
            for (int j = 1; j < nf; ++j) {
                const double* c = fixed_chain + (long long)j * 9;
                double g[9];
                bool ok = base && (fixed_conn == nullptr || fixed_conn[j] != 0);
                if (ok) {
                    for (int row = 0; row < 3; ++row)
                        for (int col = 0; col < 3; ++col)
                            g[row * 3 + col] = c0i[row * 3] * c[col] + c0i[row * 3 + 1] * c[3 + col] + c0i[row * 3 + 2] * c[6 + col];
                    nm_renormalise(g);
                    for (int i = 0; i < 9; ++i) ok = ok && isfinite(g[i]);
                }
                for (int i = 0; i < 9; ++i) G[(long long)j * 9 + i] = ok ? g[i] : G[(long long)(j - 1) * 9 + i];
                conn[j] = ok;
            }
        }
        for (int k = nf; k < n; ++k) {
            int found = 0;
            for (int d = 1; d <= span && d <= k && !found; ++d) {
                const int l = adj_link(k - d, d, n);
                if (!conn[k - d] || !usable(l)) continue;
                double r[9], g[9];
                nm_chain_step(H_links + (long long)l * 9, true, r);
                const double* a = G + (long long)(k - d) * 9;
                for (int row = 0; row < 3; ++row)
                    for (int c = 0; c < 3; ++c) g[row * 3 + c] = a[row * 3] * r[c] + a[row * 3 + 1] * r[3 + c] + a[row * 3 + 2] * r[6 + c];
                nm_renormalise(g);
                for (int i = 0; i < 9; ++i) G[(long long)k * 9 + i] = g[i];
                found = 1;
            }
            if (!found)
                for (int i = 0; i < 9; ++i) G[(long long)k * 9 + i] = G[(long long)(k - 1) * 9 + i];
            conn[k] = found;
        }
        AdjState st;
        st.lambda = -1.0; st.cost = st.cost0 = 0.0;
        st.first = 1; st.done = 0; st.accepted = 0; st.nonfinite = 0;
        *state = st;
    }
    __syncthreads();
    for (int k = tid; k < n; k += 256) {
        double th[NP];
        if (k == 0) adj_identity<KIND>(th);
        else {
            double Gn[9];
            adj_conj(geo, G + (long long)k * 9, Gn, true);
            adj_params<KIND>(Gn, th);
        }
        for (int i = 0; i < NP; ++i) x_cur[k * NP + i] = x_eval[k * NP + i] = th[i];
    }
    for (int l = tid; l < L; l += 256) {
        int t, d;
        nm_link_decode(l, n, t, d);
        used[l] = t + d >= nf && conn[t] && conn[t + d] && usable(l);
    }
}

// One CTA per (link, slice): the slice's share of the link's J^T J blocks, J^T r and cost at x_eval.  A pass stages
// kAdjThreads correspondences (residual and projection derivatives) in shared memory; thread e then adds entry e of
// every staged point in index order, so the sums have a fixed order.  Entry e is +/-(a1 b1 + a2 b2) of staged values.
// COST 0 (mosaic) stages dpi(Gn_u b) / dth_u, so the (t, u) block and J^T r of u are negated; COST 1 (transfer) stages
// dr / dth_u itself and sets state->nonfinite for a point that makes the cost +inf (state is not __restrict__: the
// kernel reads state->done and a transfer build writes the flag).
template <int KIND, int COST>
__global__ void __launch_bounds__(kAdjThreads) adjust_build_kernel(const Pairs P, const unsigned char* __restrict__ masks, int n,
                                                                   AdjGeom geo, const int* __restrict__ used,
                                                                   const double* __restrict__ x_eval, AdjState* state,
                                                                   double* __restrict__ partial)
{
    constexpr int NP = AdjFam<KIND>::P, E = AdjFam<KIND>::E, W = AdjFam<KIND>::W;
    constexpr int NE = (E + kAdjThreads - 1) / kAdjThreads;
    __shared__ double sp[kAdjThreads * W];
    __shared__ unsigned char sv[kAdjThreads];
    const int l = blockIdx.x, slice = blockIdx.y, tid = threadIdx.x;
    if (state->done || !used[l]) return;
    int t, d;
    nm_link_decode(l, n, t, d);
    double tht[NP], thu[NP];
    for (int i = 0; i < NP; ++i) { tht[i] = x_eval[t * NP + i]; thu[i] = x_eval[(t + d) * NP + i]; }
    double Gi[9], M[9];                                      // transfer: Gn_u^-1 and Gn_u^-1 Gn_t of this link
    if constexpr (COST == 1) {
        double Gt[9], Gu[9];
        adj_matrix<KIND>(tht, Gt);
        adj_matrix<KIND>(thu, Gu);
        nm_inv3d(Gu, nm_det3d(Gu), Gi);
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) M[r * 3 + c] = Gi[r * 3] * Gt[c] + Gi[r * 3 + 1] * Gt[3 + c] + Gi[r * 3 + 2] * Gt[6 + c];
    }
    // entries owned by this thread: (a1, b1, a2, b2, negate)
    int ea[NE][4];
    bool neg[NE];
    for (int r = 0; r < NE; ++r) {
        const int e = tid + r * kAdjThreads;
        int a1 = 0, b1 = 0, a2 = 1, b2 = 1;
        bool ng = false;
        const int ot = 2, ovt = 2 + NP, ou = 2 + 2 * NP, ovu = 2 + 3 * NP;    // du_t, dv_t, du_u, dv_u
        if (e < NP * NP) { const int i = e / NP, j = e % NP; a1 = ot + i; b1 = ot + j; a2 = ovt + i; b2 = ovt + j; }
        else if (e < 2 * NP * NP) { const int i = (e - NP * NP) / NP, j = e % NP; a1 = ou + i; b1 = ou + j; a2 = ovu + i; b2 = ovu + j; }
        else if (e < 3 * NP * NP) { const int i = (e - 2 * NP * NP) / NP, j = e % NP; a1 = ot + i; b1 = ou + j; a2 = ovt + i; b2 = ovu + j; ng = COST == 0; }
        else if (e < 3 * NP * NP + NP) { const int i = e - 3 * NP * NP; a1 = ot + i; b1 = 0; a2 = ovt + i; b2 = 1; }
        else if (e < 3 * NP * NP + 2 * NP) { const int i = e - 3 * NP * NP - NP; a1 = ou + i; b1 = 0; a2 = ovu + i; b2 = 1; ng = COST == 0; }
        ea[r][0] = a1; ea[r][1] = b1; ea[r][2] = a2; ea[r][3] = b2;
        neg[r] = ng;
    }
    double acc[NE];
    for (int r = 0; r < NE; ++r) acc[r] = 0.0;
    const int cnt = pair_n(P, l), len = (cnt + kAdjSlices - 1) / kAdjSlices;
    const int lo = slice * len, hi = min(cnt, lo + len);
    const long long off = (long long)l * P.stride;
    const unsigned char* __restrict__ mask = masks + (long long)l * P.max_pts;
    bool bad = false;
    for (int base = lo; base < hi; base += kAdjThreads) {
        const int i = base + tid;
        const bool ok = i < hi && mask[i] != 0;
        if (ok) {
            double* q = sp + tid * W;
            const double2 a = geo.norm(P.sx[off + i], P.sy[off + i]), b = geo.norm(P.dx[off + i], P.dy[off + i]);
            if constexpr (COST == 0) {
                double Ut, Vt, Uu, Vu;
                adj_project<KIND>(tht, a.x, a.y, Ut, Vt, q + 2, q + 2 + NP);
                adj_project<KIND>(thu, b.x, b.y, Uu, Vu, q + 2 + 2 * NP, q + 2 + 3 * NP);
                q[0] = Ut - Uu;
                q[1] = Vt - Vu;
            } else if (!adj_transfer<KIND>(Gi, M, a, b, q))
                bad = true;
        }
        sv[tid] = ok;
        __syncthreads();
        const int np = min(kAdjThreads, hi - base);
        for (int k = 0; k < np; ++k) {
            if (!sv[k]) continue;
            const double* q = sp + k * W;
#pragma unroll
            for (int r = 0; r < NE; ++r) acc[r] += q[ea[r][0]] * q[ea[r][1]] + q[ea[r][2]] * q[ea[r][3]];
        }
        __syncthreads();
    }
    for (int r = 0; r < NE; ++r) {
        const int e = tid + r * kAdjThreads;
        if (e < E) partial[((long long)l * kAdjSlices + slice) * E + e] = neg[r] ? -acc[r] : acc[r];
    }
    if constexpr (COST == 1)
        if (bad) state->nonfinite = 1;
}

// One CTA: the Levenberg-Marquardt step.  Link totals (slices in order), the cost at x_eval (links in index order, +inf
// when the build flagged a point); x_eval is accepted when it is the first point or lowers the cost (lambda / 10), else
// rejected (lambda * 10).  A +inf cost at the first point ends the run there: the window keeps its initial poses.  After an
// acceptance the banded normal equations of the unknowns (frame-major, half-bandwidth bw = P (span + 1) - 1; the rows
// of a disconnected or fixed frame k < nf are the identity with zero right-hand side) are assembled in link index order.  Unless the
// run is over, (J^T J + lambda I) delta = -J^T r is solved by a banded Cholesky factorisation -- the last bw + 1 rows of
// the factor kept in shared memory, the forward substitution folded into it, the back substitution by warp 0 -- and
// x_eval = x_cur + delta.  A failed factorisation counts as a rejection.
template <int KIND>
__global__ void __launch_bounds__(kAdjSolveThreads) adjust_solve_kernel(int n, int span, int nf, const int* __restrict__ used,
                                                                        const int* __restrict__ conn, const double* __restrict__ partial,
                                                                        double* __restrict__ link_tot, double* __restrict__ A,
                                                                        double* __restrict__ rhs, double* __restrict__ U,
                                                                        double* __restrict__ x_cur, double* __restrict__ x_eval,
                                                                        AdjState* state, int last)
{
    constexpr int NP = AdjFam<KIND>::P, E = AdjFam<KIND>::E;
    extern __shared__ double sm[];
    __shared__ int s_accept, s_stop, s_fail;
    const int tid = threadIdx.x, L = nm_span_links(n, span), m = (n - 1) * NP, bw = NP * (span + 1) - 1, bw1 = bw + 1;
    double* W = sm;                                          // [bw1][bw1] rows of the factor, row k at slot k % bw1
    double* tmp = W + bw1 * bw1;                             // [bw1 + 1]
    double* y = tmp + bw1 + 1;                               // [m] forward, then back substitution
    if (state->done) return;
    for (int idx = tid; idx < L * E; idx += kAdjSolveThreads) {
        const int l = idx / E, e = idx - l * E;
        if (!used[l]) continue;
        const double* q = partial + (long long)l * kAdjSlices * E + e;
        double s = q[0];
        for (int sl = 1; sl < kAdjSlices; ++sl) s += q[sl * E];
        link_tot[idx] = s;
    }
    __syncthreads();
    if (tid == 0) {
        double c = 0.0;
        for (int l = 0; l < L; ++l)
            if (used[l]) c += link_tot[(long long)l * E + E - 1];
        AdjState st = *state;
        if (st.nonfinite) c = INFINITY;
        bool accept = false;
        if (st.first) { accept = true; st.cost0 = c; st.first = 0; if (st.nonfinite) st.done = 1; }
        else if (c < st.cost) {
            accept = true;
            if (st.cost - c < 1e-12 * st.cost) st.done = 1;
            st.lambda *= 0.1;
            ++st.accepted;
        } else {
            st.lambda *= 10.0;
            if (st.lambda > 1e16) st.done = 1;
        }
        if (accept) st.cost = c;
        st.nonfinite = 0;
        *state = st;
        s_accept = accept;
        s_stop = st.done || last;
    }
    __syncthreads();
    const bool accept = s_accept;
    if (accept)
        for (int i = tid; i < n * NP; i += kAdjSolveThreads) x_cur[i] = x_eval[i];
    if (s_stop) return;
    if (accept) {
        for (long long idx = tid; idx < (long long)m * bw1; idx += kAdjSolveThreads) {
            const int i = (int)(idx / bw1), c = (int)(idx - (long long)i * bw1), j = i + c;
            double v = 0.0;
            if (j < m) {
                const int k = i / NP + 1, a = i % NP, k2 = j / NP + 1, b = j % NP, dd = k2 - k;
                if (k < nf || !conn[k] || !conn[k2]) v = c == 0 ? 1.0 : 0.0;   // k2 >= k is free if k is
                else if (dd == 0) {
                    for (int d = 1; d <= span; ++d) {
                        if (k - d >= 0) { const int l = adj_link(k - d, d, n); if (used[l]) v += link_tot[(long long)l * E + NP * NP + a * NP + b]; }
                        if (k + d < n) { const int l = adj_link(k, d, n); if (used[l]) v += link_tot[(long long)l * E + a * NP + b]; }
                    }
                } else if (dd <= span) {
                    const int l = adj_link(k, dd, n);
                    if (used[l]) v = link_tot[(long long)l * E + 2 * NP * NP + a * NP + b];
                }
            }
            A[idx] = v;
        }
        for (int i = tid; i < m; i += kAdjSolveThreads) {
            const int k = i / NP + 1, a = i % NP;
            double v = 0.0;
            if (k >= nf && conn[k])
                for (int d = 1; d <= span; ++d) {
                    if (k - d >= 0) { const int l = adj_link(k - d, d, n); if (used[l]) v += link_tot[(long long)l * E + 3 * NP * NP + NP + a]; }
                    if (k + d < n) { const int l = adj_link(k, d, n); if (used[l]) v += link_tot[(long long)l * E + 3 * NP * NP + a]; }
                }
            rhs[i] = v;
        }
        __syncthreads();
        if (tid == 0 && state->lambda < 0.0) {
            double mx = 0.0;
            for (int i = 0; i < m; ++i)
                if (i / NP + 1 >= nf && conn[i / NP + 1]) mx = fmax(mx, A[(long long)i * bw1]);
            state->lambda = mx > 0.0 ? 1e-3 * mx : 1e-3;
        }
        __syncthreads();
    }
    for (;;) {
        const double lambda = state->lambda;
        bool fail = false;
        for (int j = 0; j < m && !fail; ++j) {
            if (tid <= bw) {
                const int i = j + tid;
                if (i < m) {
                    double s = A[(long long)j * bw1 + tid] + (tid == 0 ? lambda : 0.0);
                    const int k0 = max(0, i - bw);
                    int slot = k0 % bw1;
                    for (int k = k0; k < j; ++k) {
                        s -= W[slot * bw1 + (j - k)] * W[slot * bw1 + (i - k)];
                        slot = slot + 1 == bw1 ? 0 : slot + 1;
                    }
                    tmp[tid] = s;
                }
            } else if (tid == bw1) {
                double s = -rhs[j];
                const int k0 = max(0, j - bw);
                int slot = k0 % bw1;
                for (int k = k0; k < j; ++k) {
                    s -= W[slot * bw1 + (j - k)] * y[k];
                    slot = slot + 1 == bw1 ? 0 : slot + 1;
                }
                tmp[bw1] = s;
            }
            __syncthreads();
            const double dj = tmp[0];
            fail = !(dj > 0.0) || !isfinite(dj);
            if (!fail) {
                const double r = sqrt(dj);
                if (tid <= bw && j + tid < m) {
                    const double v = tid == 0 ? r : tmp[tid] / r;
                    W[(j % bw1) * bw1 + tid] = v;
                    U[(long long)j * bw1 + tid] = v;
                } else if (tid == bw1) y[j] = tmp[bw1] / r;
            }
            __syncthreads();
        }
        if (!fail && tid < 32) {
            // back substitution U delta = y, in place; lane c handles the columns i + 1 + c + 32 q
            for (int i = m - 1; i >= 0; --i) {
                double s = 0.0;
                for (int c = 1 + tid; c <= bw && i + c < m; c += 32) s += U[(long long)i * bw1 + c] * y[i + c];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                const double v = (y[i] - s) / U[(long long)i * bw1];
                __syncwarp();
                if (tid == 0) y[i] = v;
                __syncwarp();
                if (!isfinite(v)) fail = true;
            }
            if (tid == 0) s_fail = fail;
        } else if (tid == 0) s_fail = fail;
        __syncthreads();
        fail = s_fail;
        if (!fail) {
            for (int i = tid; i < n * NP; i += kAdjSolveThreads) {
                const int k = i / NP;
                x_eval[i] = (k < nf || !conn[k]) ? x_cur[i] : x_cur[i] + y[i - NP];
            }
            return;
        }
        if (tid == 0) {
            state->lambda *= 10.0;
            if (state->lambda > 1e16) state->done = 1;
        }
        __syncthreads();
        if (state->done) return;
    }
}

// One CTA per pair p: H_out[p] = G_(p+1)^-1 G_p rounded to float (divided by its [8]) and status {1, inliers of it on link
// (p, 1), LM steps accepted} when frame p + 1 is connected; H_in[p] and {0, 0, 0} otherwise (nm_mosaic_place_f32 then
// keeps frame p + 1 at G_p).  chain_out[p + 1] (and [0] by CTA 0) = G; CTA 0 writes the report.
template <int KIND>
__global__ void __launch_bounds__(256) adjust_finish_kernel(const Pairs P, float thr, int n, int span, AdjGeom geo,
                                                            const float* H_in, const int* __restrict__ conn,
                                                            const int* __restrict__ used, const int* __restrict__ npts,
                                                            const double* __restrict__ x_cur, const AdjState* __restrict__ state,
                                                            float* H_out, int* status_out, double* __restrict__ chain_out,
                                                            double* __restrict__ report)
{
    constexpr int NP = AdjFam<KIND>::P;
    __shared__ float Hs[9];
    __shared__ int s_cnt;
    const int p = blockIdx.x, k = p + 1, tid = threadIdx.x;
    if (tid == 0) {
        // a disconnected frame sits at the adjusted pose of its nearest connected predecessor
        int ep = p, ek = k;
        while (!conn[ep]) --ep;
        if (!conn[ek]) ek = ep;
        double thp[NP], thk[NP], Gp[9], Gk[9], Gki[9], Mn[9], M[9];
        for (int i = 0; i < NP; ++i) { thp[i] = x_cur[ep * NP + i]; thk[i] = x_cur[ek * NP + i]; }
        adj_matrix<KIND>(thp, Gp);
        adj_matrix<KIND>(thk, Gk);
        if (chain_out) {
            double C[9];
            adj_conj(geo, Gk, C, false);
            for (int i = 0; i < 9; ++i) chain_out[(long long)k * 9 + i] = C[i];
            if (p == 0) for (int i = 0; i < 9; ++i) chain_out[i] = (i % 4 == 0) ? 1.0 : 0.0;
        }
        nm_inv3d(Gk, nm_det3d(Gk), Gki);
        for (int r = 0; r < 3; ++r)
            for (int c = 0; c < 3; ++c) Mn[r * 3 + c] = Gki[r * 3] * Gp[c] + Gki[r * 3 + 1] * Gp[3 + c] + Gki[r * 3 + 2] * Gp[6 + c];
        adj_conj(geo, Mn, M, false);
        for (int i = 0; i < 9; ++i) Hs[i] = conn[k] ? (float)(M[i] / M[8]) : H_in[(long long)p * 9 + i];
        s_cnt = 0;
        if (p == 0 && report) {
            long long pts = 0;
            int links = 0;
            for (int l = 0; l < nm_span_links(n, span); ++l)
                if (used[l]) { pts += npts[l]; ++links; }
            const double scale = 1.0 / (geo.s * geo.s * (double)(pts > 0 ? pts : 1));
            report[0] = state->cost0 * scale;
            report[1] = state->cost * scale;
            report[2] = (double)pts;
            report[3] = (double)links;
        }
    }
    __syncthreads();
    if (!conn[k]) {
        if (tid < 9) H_out[(long long)p * 9 + tid] = Hs[tid];
        if (tid == 0) status_out[p * 3] = status_out[p * 3 + 1] = status_out[p * 3 + 2] = 0;
        return;
    }
    float H[9];
    for (int i = 0; i < 9; ++i) H[i] = Hs[i];
    const int cnt = pair_n(P, p);
    const long long off = (long long)p * P.stride;
    int c = 0;
    for (int i = tid; i < cnt; i += 256) c += transfer_inlier(H, make_float4(P.sx[off + i], P.sy[off + i], P.dx[off + i], P.dy[off + i]), thr);
    atomicAdd(&s_cnt, c);
    __syncthreads();
    if (tid < 9) H_out[(long long)p * 9 + tid] = H[tid];
    if (tid == 0) {
        status_out[p * 3] = 1;
        status_out[p * 3 + 1] = s_cnt;
        status_out[p * 3 + 2] = state->accepted;
    }
}

template <int KIND>
int adjust_chain(const Pairs& P, int cost, float thr, int n, int span, int fw, int fh, const unsigned char* masks,
                 const float* H_links, const int* link_status, int n_fixed, const double* fixed_chain, const int* fixed_conn,
                 int iterations, float* H_out, int* status_out, double* chain_out, double* report, cudaStream_t st)
{
    constexpr int NP = AdjFam<KIND>::P, E = AdjFam<KIND>::E;
    const int L = nm_span_links(n, span), m = (n - 1) * NP, bw1 = NP * (span + 1);
    const size_t smem = sizeof(double) * ((size_t)bw1 * bw1 + bw1 + 1 + m);
    static NmDeviceOnce once;
    if (once.first()) {
        NM_CUDA_TRY(cudaFuncSetAttribute(adjust_solve_kernel<KIND>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)(sizeof(double) * ((size_t)(8 * (kAdjMaxSpan + 1)) * (8 * (kAdjMaxSpan + 1)) +
                                                                 8 * (kAdjMaxSpan + 1) + 1 + (kAdjMaxFrames - 1) * 8))));
        once.done();
    }
    // one stream-ordered block: state | G | x_cur | x_eval | partial | link_tot | A | U | rhs (doubles), conn | used | npts
    const size_t nd = 8 + 9 * (size_t)n + 2 * (size_t)n * NP + (size_t)L * kAdjSlices * E + (size_t)L * E +
                      2 * (size_t)m * bw1 + (size_t)m;
    const size_t total = sizeof(double) * nd + sizeof(int) * ((size_t)n + 2 * (size_t)L);
    char* ws = nullptr;
    NM_CUDA_TRY(nm_ws_alloc(&ws, total, st));
    double* d = reinterpret_cast<double*>(ws);
    AdjState* state = reinterpret_cast<AdjState*>(d);
    double* G = d + 8;
    double* x_cur = G + 9 * (size_t)n;
    double* x_eval = x_cur + (size_t)n * NP;
    double* partial = x_eval + (size_t)n * NP;
    double* link_tot = partial + (size_t)L * kAdjSlices * E;
    double* A = link_tot + (size_t)L * E;
    double* U = A + (size_t)m * bw1;
    double* rhs = U + (size_t)m * bw1;
    int* conn = reinterpret_cast<int*>(rhs + m);
    int* used = conn + n;
    int* npts = used + L;
    const double ext = (double)(fw > fh ? fw : fh);
    const AdjGeom geo{0.5 * (fw - 1), 0.5 * (fh - 1), 2.0 / ext};
    adjust_count_kernel<<<L, 256, 0, st>>>(P, masks, npts);
    adjust_init_kernel<KIND><<<1, 256, 0, st>>>(n, span, geo, H_links, link_status, npts, n_fixed, fixed_chain, fixed_conn, G, conn,
                                                used, x_cur, x_eval, state);
    for (int it = 0; it < iterations; ++it) {
        if (cost == NM_ADJUST_MOSAIC)
            adjust_build_kernel<KIND, 0><<<dim3(L, kAdjSlices), kAdjThreads, 0, st>>>(P, masks, n, geo, used, x_eval, state, partial);
        else
            adjust_build_kernel<KIND, 1><<<dim3(L, kAdjSlices), kAdjThreads, 0, st>>>(P, masks, n, geo, used, x_eval, state, partial);
        adjust_solve_kernel<KIND><<<1, kAdjSolveThreads, smem, st>>>(n, span, n_fixed, used, conn, partial, link_tot, A, rhs, U,
                                                                     x_cur, x_eval, state, it == iterations - 1);
    }
    adjust_finish_kernel<KIND><<<n - 1, 256, 0, st>>>(P, thr, n, span, geo, H_links, conn, used, npts, x_cur, state, H_out, status_out,
                                                      chain_out, report);
    const cudaError_t e = cudaGetLastError();
    const cudaError_t f = cudaFreeAsync(ws, st);
    return nm_cuda_err(e != cudaSuccess ? e : f);
}

int min_points(int kind) { return kind == 2 ? 4 : 2; }        // ransac.cu:541, :606, :656 (translation also asks for 2)
int sample_size(int kind) { return kind == 0 ? 1 : kind == 1 ? 2 : 4; }

int launch_hypotheses(int kind, const Pairs& P, int n_pairs, const int* rand_list, int iterations, float thr, const int* state,
                      float* H_all, int* inliers, unsigned char* skip, cudaStream_t st)
{
    const dim3 grid(nm_div_up(iterations, kHypThreads), n_pairs);
    const int mp = min_points(kind);
    if (kind == 0) hypothesis_kernel<0><<<grid, kHypThreads, 0, st>>>(P, rand_list, iterations, state, mp, H_all, inliers, skip);
    else if (kind == 1) hypothesis_kernel<1><<<grid, kHypThreads, 0, st>>>(P, rand_list, iterations, state, mp, H_all, inliers, skip);
    else hypothesis_kernel<2><<<grid, kHypThreads, 0, st>>>(P, rand_list, iterations, state, mp, H_all, inliers, skip);
    NM_LAUNCH_CHECK();
    const dim3 sg(nm_div_up(iterations, kScoreThreads), nm_div_up(P.max_pts, kScorePts), n_pairs);
    score_kernel<<<sg, kScoreThreads, 0, st>>>(P, H_all, skip, iterations, thr, inliers);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int ransac_batch(int kind, const Pairs& P, int n_pairs, float thr, int iterations, unsigned long long seed, float* homographies,
                 int* status, cudaStream_t st)
{
    const int m = sample_size(kind), mp = min_points(kind);
    const long long draws = (long long)iterations * m;
    if (draws >= (1LL << 31) || (long long)n_pairs * iterations >= (1LL << 31) || n_pairs > 65535) return NM_ERR_INVALID;
    // one stream-ordered block: valid lists | states | rand lists | homographies | inliers | skip flags
    const size_t np = (size_t)n_pairs;
    const size_t o_valid = 0, o_state = o_valid + sizeof(int) * np * (size_t)P.max_pts, o_rand = o_state + 16 * np,
                 o_H = o_rand + sizeof(int) * np * (size_t)draws, o_inl = o_H + sizeof(float) * 9 * np * (size_t)iterations,
                 o_skip = o_inl + sizeof(int) * np * (size_t)iterations, total = o_skip + np * (size_t)iterations;
    char* ws = nullptr;
    NM_CUDA_TRY(nm_ws_alloc(&ws, total, st));
    int* valid = reinterpret_cast<int*>(ws + o_valid);
    int* state = reinterpret_cast<int*>(ws + o_state);
    int* rand_list = reinterpret_cast<int*>(ws + o_rand);
    float* H_all = reinterpret_cast<float*>(ws + o_H);
    int* inl = reinterpret_cast<int*>(ws + o_inl);
    unsigned char* skip = reinterpret_cast<unsigned char*>(ws + o_skip);
    valid_list_kernel<<<n_pairs, 1024, 0, st>>>(P, valid, state);
    draw_kernel<<<dim3(nm_div_up((int)draws, 256), n_pairs), 256, 0, st>>>(valid, state, P.max_pts, mp, seed, (int)draws, rand_list);
    int rc = cudaGetLastError() == cudaSuccess ? NM_OK : NM_ERR_CUDA_BASE;
    if (rc == NM_OK) rc = launch_hypotheses(kind, P, n_pairs, rand_list, iterations, thr, state, H_all, inl, skip, st);
    if (rc == NM_OK) {
        select_kernel<<<n_pairs, 256, 0, st>>>(inl, H_all, iterations, state, mp, homographies, status);
        rc = cudaGetLastError() == cudaSuccess ? NM_OK : NM_ERR_CUDA_BASE;
    }
    NM_CUDA_TRY(cudaFreeAsync(ws, st));
    return rc;
}

} // namespace

extern "C" int nm_align_points_f32(const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                                   float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y,
                                   const int* matches, int num_pts, nm_stream_t stream)
{
    if (num_pts < 0) return NM_ERR_INVALID;
    if (num_pts == 0) return NM_OK;
    if (!src_x || !src_y || !dst_x || !dst_y || !c_src_x || !c_src_y || !c_dst_x || !c_dst_y || !matches) return NM_ERR_INVALID;
    align_kernel<<<nm_div_up(num_pts, 256), 256, 0, (cudaStream_t)stream>>>(src_x, src_y, dst_x, dst_y, c_src_x, c_src_y,
                                                                          c_dst_x, c_dst_y, matches, num_pts);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_align_pairs_span_f32(const float* x, const float* y, const int* matches, const int* counts_dev, int n_frames,
                                       int capacity, int span, float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y,
                                       nm_stream_t stream)
{
    if (!x || !y || !matches || !counts_dev || !c_src_x || !c_src_y || !c_dst_x || !c_dst_y || n_frames < 2 || capacity <= 0)
        return NM_ERR_INVALID;
    if (span < 1 || span > 8 || span > n_frames - 1 || nm_span_links(n_frames, span) > 65535) return NM_ERR_INVALID;
    align_pairs_kernel<<<dim3(nm_div_up(capacity, 256), nm_span_links(n_frames, span)), 256, 0, (cudaStream_t)stream>>>(
        x, y, matches, counts_dev, n_frames, capacity, c_src_x, c_src_y, c_dst_x, c_dst_y);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_align_pairs_f32(const float* x, const float* y, const int* matches, const int* counts_dev, int n_frames,
                                  int capacity, float* c_src_x, float* c_src_y, float* c_dst_x, float* c_dst_y,
                                  nm_stream_t stream)
{
    return nm_align_pairs_span_f32(x, y, matches, counts_dev, n_frames, capacity, 1, c_src_x, c_src_y, c_dst_x, c_dst_y, stream);
}

extern "C" int nm_ransac_hypotheses_f32(int kind, const float* src_x, const float* src_y, const float* dst_x,
                                        const float* dst_y, int num_pts, const int* rand_list, int iterations,
                                        float inlier_threshold, float* homographies, int* inliers, nm_stream_t stream)
{
    if (kind < 0 || kind > 2 || num_pts <= 0 || iterations <= 0) return NM_ERR_INVALID;
    if (!src_x || !src_y || !dst_x || !dst_y || !rand_list || !homographies || !inliers) return NM_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    unsigned char* skip = nullptr;
    NM_CUDA_TRY(nm_ws_alloc(&skip, (size_t)iterations, st));
    const Pairs P{src_x, src_y, dst_x, dst_y, 0, nullptr, num_pts};
    const int rc = launch_hypotheses(kind, P, 1, rand_list, iterations, inlier_threshold, nullptr, homographies, inliers, skip, st);
    NM_CUDA_TRY(cudaFreeAsync(skip, st));
    return rc;
}

extern "C" int nm_ransac_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                             int num_pts, float inlier_threshold, int iterations, unsigned long long seed,
                             float* homography, int* status, nm_stream_t stream)
{
    if (kind < 0 || kind > 2 || num_pts <= 0 || iterations <= 0) return NM_ERR_INVALID;
    if (!src_x || !src_y || !dst_x || !dst_y || !homography || !status) return NM_ERR_INVALID;
    const Pairs P{src_x, src_y, dst_x, dst_y, 0, nullptr, num_pts};
    return ransac_batch(kind, P, 1, inlier_threshold, iterations, seed, homography, status, (cudaStream_t)stream);
}

extern "C" int nm_ransac_batch_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                                   long long pair_stride, const int* counts, int max_pts, int n_pairs, float inlier_threshold,
                                   int iterations, unsigned long long seed, float* homographies, int* status, nm_stream_t stream)
{
    if (kind < 0 || kind > 2 || max_pts <= 0 || n_pairs <= 0 || iterations <= 0 || pair_stride < 0) return NM_ERR_INVALID;
    if (!src_x || !src_y || !dst_x || !dst_y || !homographies || !status) return NM_ERR_INVALID;
    const Pairs P{src_x, src_y, dst_x, dst_y, pair_stride, counts, max_pts};
    return ransac_batch(kind, P, n_pairs, inlier_threshold, iterations, seed, homographies, status, (cudaStream_t)stream);
}

extern "C" int nm_ransac_refine_batch_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                                          long long pair_stride, const int* counts, int max_pts, int n_pairs,
                                          float inlier_threshold, const float* H_in, const int* status_in, int rounds,
                                          float* H_out, int* status_out, unsigned char* inlier_mask, nm_stream_t stream)
{
    if (kind < 0 || kind > 2 || max_pts <= 0 || n_pairs <= 0 || rounds < 0 || pair_stride < 0) return NM_ERR_INVALID;
    if (!src_x || !src_y || !dst_x || !dst_y || !H_in || !H_out || !status_out) return NM_ERR_INVALID;
    const Pairs P{src_x, src_y, dst_x, dst_y, pair_stride, counts, max_pts};
    cudaStream_t st = (cudaStream_t)stream;
    if (kind == 0) refine_kernel<0><<<n_pairs, kRefineThreads, 0, st>>>(P, inlier_threshold, H_in, status_in, rounds, H_out, status_out, inlier_mask);
    else if (kind == 1) refine_kernel<1><<<n_pairs, kRefineThreads, 0, st>>>(P, inlier_threshold, H_in, status_in, rounds, H_out, status_out, inlier_mask);
    else refine_kernel<2><<<n_pairs, kRefineThreads, 0, st>>>(P, inlier_threshold, H_in, status_in, rounds, H_out, status_out, inlier_mask);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_ransac_adjust_chain_fixed_f32(int kind, int cost, const float* src_x, const float* src_y, const float* dst_x,
                                                const float* dst_y, long long pair_stride, const int* counts, int max_pts,
                                                float inlier_threshold, int n_frames, int span, int frame_w, int frame_h,
                                                const unsigned char* masks, const float* H_links, const int* link_status,
                                                int n_fixed, const double* fixed_chain, const int* fixed_conn, int iterations,
                                                float* H_out, int* status_out, double* chain_out, double* report_out,
                                                nm_stream_t stream)
{
    if (kind < 0 || kind > 2 || max_pts <= 0 || pair_stride < 0 || iterations < 1 || frame_w <= 0 || frame_h <= 0) return NM_ERR_INVALID;
    if (cost != NM_ADJUST_MOSAIC && cost != NM_ADJUST_TRANSFER) return NM_ERR_INVALID;
    if (n_frames < 2 || n_frames > kAdjMaxFrames || span < 1 || span > kAdjMaxSpan || span >= n_frames) return NM_ERR_INVALID;
    if (n_fixed < 1 || n_fixed >= n_frames || (n_fixed > 1 && !fixed_chain)) return NM_ERR_INVALID;
    if (!src_x || !src_y || !dst_x || !dst_y || !masks || !H_links || !link_status || !H_out || !status_out) return NM_ERR_INVALID;
    const Pairs P{src_x, src_y, dst_x, dst_y, pair_stride, counts, max_pts};
    const cudaStream_t st = (cudaStream_t)stream;
    if (kind == 0)
        return adjust_chain<0>(P, cost, inlier_threshold, n_frames, span, frame_w, frame_h, masks, H_links, link_status, n_fixed,
                               fixed_chain, fixed_conn, iterations, H_out, status_out, chain_out, report_out, st);
    if (kind == 1)
        return adjust_chain<1>(P, cost, inlier_threshold, n_frames, span, frame_w, frame_h, masks, H_links, link_status, n_fixed,
                               fixed_chain, fixed_conn, iterations, H_out, status_out, chain_out, report_out, st);
    return adjust_chain<2>(P, cost, inlier_threshold, n_frames, span, frame_w, frame_h, masks, H_links, link_status, n_fixed,
                           fixed_chain, fixed_conn, iterations, H_out, status_out, chain_out, report_out, st);
}

extern "C" int nm_ransac_adjust_chain_cost_f32(int kind, int cost, const float* src_x, const float* src_y, const float* dst_x,
                                               const float* dst_y, long long pair_stride, const int* counts, int max_pts,
                                               float inlier_threshold, int n_frames, int span, int frame_w, int frame_h,
                                               const unsigned char* masks, const float* H_links, const int* link_status,
                                               int iterations, float* H_out, int* status_out, double* chain_out, double* report_out,
                                               nm_stream_t stream)
{
    return nm_ransac_adjust_chain_fixed_f32(kind, cost, src_x, src_y, dst_x, dst_y, pair_stride, counts, max_pts, inlier_threshold,
                                            n_frames, span, frame_w, frame_h, masks, H_links, link_status, 1, nullptr, nullptr,
                                            iterations, H_out, status_out, chain_out, report_out, stream);
}

extern "C" int nm_ransac_adjust_chain_f32(int kind, const float* src_x, const float* src_y, const float* dst_x, const float* dst_y,
                                          long long pair_stride, const int* counts, int max_pts, float inlier_threshold,
                                          int n_frames, int span, int frame_w, int frame_h, const unsigned char* masks,
                                          const float* H_links, const int* link_status, int iterations, float* H_out,
                                          int* status_out, double* chain_out, double* report_out, nm_stream_t stream)
{
    return nm_ransac_adjust_chain_cost_f32(kind, NM_ADJUST_MOSAIC, src_x, src_y, dst_x, dst_y, pair_stride, counts, max_pts,
                                           inlier_threshold, n_frames, span, frame_w, frame_h, masks, H_links, link_status,
                                           iterations, H_out, status_out, chain_out, report_out, stream);
}
