// nm_mosaic.cu -- the step AFTER registration (SURVEY.md 8f rank 4): perspective coordinate maps, resampling
// through the caller's textures and the weighted blend of a warped frame into the mosaic canvas.
//
// Replaces resample_perspective_transform (gpu/kernels/resample.cu:119-219, :221-233), resample_mask
// (:67-81, :236-244) and transform_blend (:7-65, :246-258).  The texture objects are the caller's (CudaTex2D:
// linear filtering, border addressing, un-normalised coordinates), so the filtered samples are produced by
// the same texture unit as in the reference; the arithmetic around them is written in the reference's
// order.  Flat 1-D grids: every kernel here is one independent HBM-bound pass over the output pixels.
//
// The mosaic of a registered frame stream (nm_mosaic_*): place_kernel chains the pairwise homographies into
// frame -> mosaic transforms and lays the frames out on a canvas; blend_stream_kernel blends a chunk of frames
// in one pass over the canvas, bitwise what one transform_blend call per frame, in frame order, produces.
#include "nm_chain.cuh"
#include <climits>
#include <cstdint>
#include <cstring>
#include <new>
#include <vector>

namespace {

struct Mat3 { float m[9]; };

// The reference's a*x + b*y + c and a*b - c*d as its build contracts them (established against the vectors
// the reference produced, tests/golden/mosaic_128x90.npz): the first product is fused into the sum, the second
// one is rounded on its own.  Written with explicit intrinsics so that this build cannot choose differently.
__device__ __forceinline__ float lin3(float a, float x, float b, float y, float c)
{
    return __fadd_rn(__fmaf_rn(a, x, __fmul_rn(b, y)), c);
}
__device__ __forceinline__ float det2(float a, float b, float c, float d)     // a*b - c*d
{
    return __fmaf_rn(a, b, -__fmul_rn(c, d));
}

// the inverse of apply_perspective_inverse (resample.cu:133-150), evaluated by every thread from the same
// nine floats (the reference lets thread 0 of each block do it: same values)
__device__ __forceinline__ Mat3 invert3(const float* __restrict__ t)
{
    Mat3 r;
    const float det = __fmaf_rn(t[2], det2(t[3], t[7], t[4], t[6]),
                                __fmaf_rn(t[0], det2(t[4], t[8], t[7], t[5]), -__fmul_rn(t[1], det2(t[3], t[8], t[5], t[6]))));
    const float invdet = 1 / det;
    r.m[0] = __fmul_rn(det2(t[4], t[8], t[7], t[5]), invdet);
    r.m[1] = __fmul_rn(det2(t[2], t[7], t[1], t[8]), invdet);
    r.m[2] = __fmul_rn(det2(t[1], t[5], t[2], t[4]), invdet);
    r.m[3] = __fmul_rn(det2(t[5], t[6], t[3], t[8]), invdet);
    r.m[4] = __fmul_rn(det2(t[0], t[8], t[2], t[6]), invdet);
    r.m[5] = __fmul_rn(det2(t[3], t[2], t[0], t[5]), invdet);
    r.m[6] = __fmul_rn(det2(t[3], t[7], t[6], t[4]), invdet);
    r.m[7] = __fmul_rn(det2(t[6], t[1], t[0], t[7]), invdet);
    r.m[8] = __fmul_rn(det2(t[0], t[4], t[3], t[1]), invdet);
    return r;
}

// apply_perspective / apply_perspective_inverse (resample.cu:119-191) fused with resample_2D<uchar4> (:83-102)
template <bool INVERSE>
__global__ void __launch_bounds__(256) perspective_resample_kernel(uchar4* __restrict__ result, cudaTextureObject_t tex, int width,
                                                                   int height, float* __restrict__ x_pos, float* __restrict__ y_pos,
                                                                   const float* __restrict__ mat3x3)
{
    __shared__ float t[9];
    if (threadIdx.x == 0) {
        if (INVERSE) {
            const Mat3 inv = invert3(mat3x3);
            for (int i = 0; i < 9; ++i) t[i] = inv.m[i];
        } else {
            for (int i = 0; i < 9; ++i) t[i] = mat3x3[i];
        }
    }
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)width * height) return;
    const int y = (int)(i / width), x = (int)(i - (long long)y * width);
    const float xf = (float)x, yf = (float)y;
    const float x_p = lin3(t[0], xf, t[1], yf, t[2]);
    const float y_p = lin3(t[3], xf, t[4], yf, t[5]);
    const float s_p = lin3(t[6], xf, t[7], yf, t[8]);
    const float xs = __fdiv_rn(x_p, s_p), ys = __fdiv_rn(y_p, s_p);
    x_pos[i] = xs;
    y_pos[i] = ys;
    const float4 res = tex2D<float4>(tex, xs + 0.5f, ys + 0.5f);
    uchar4 o;
    o.x = (unsigned char)(res.x * 255.9999f);
    o.y = (unsigned char)(res.y * 255.9999f);
    o.z = (unsigned char)(res.z * 255.9999f);
    o.w = (unsigned char)(res.w * 255.9999f);
    result[i] = o;
}

// resample_mask_2D (resample.cu:67-81)
__global__ void __launch_bounds__(256) resample_mask_kernel(unsigned char* __restrict__ result, cudaTextureObject_t tex, long long n,
                                                            const float* __restrict__ x, const float* __restrict__ y, float lower_limit)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float res = tex2D<float>(tex, x[i] + 0.5f, y[i] + 0.5f);
    if (res <= lower_limit) result[i] = 0;
    else result[i] = res * 255.999f;
}

// One canvas pixel of transform_and_blend (resample.cu:7-65), in two halves that the per-frame kernel and the
// stream kernel both call, so that the two agree bit for bit by construction.  blend_sample: the warp of
// canvas-local pixel (x, y) through t and the three texture reads; false when the pixel takes no part (beyond
// the frame's far edges or outside the mask).  blend_update: the running weighted average on the canvas pixel
// and weight held in registers.  Split in two so that the per-frame kernel keeps the reference's memory
// accesses: it reads the canvas weight only for a taking part pixel, and the canvas pixel only when that
// weight is non-zero.
__device__ __forceinline__ bool blend_sample(int x, int y, const float* t, int fw, int fh, cudaTextureObject_t frame,
                                             cudaTextureObject_t mask, cudaTextureObject_t frame_wts, float4& res, float& new_weight)
{
    const float xf = (float)x, yf = (float)y;
    const float s_p = lin3(t[6], xf, t[7], yf, t[8]);
    const float x_p = __fdiv_rn(lin3(t[0], xf, t[1], yf, t[2]), s_p);
    const float y_p = __fdiv_rn(lin3(t[3], xf, t[4], yf, t[5]), s_p);
    if (x_p >= fw || y_p >= fh) return false;
    res = tex2D<float4>(frame, x_p + 0.5f, y_p + 0.5f);
    const float in_mask = tex2D<float>(mask, x_p + 0.5f, y_p + 0.5f);
    if (in_mask <= 0.5) return false;
    new_weight = tex2D<float>(frame_wts, x_p + 0.5f, y_p + 0.5f);
    return true;
}

__device__ __forceinline__ void blend_update(const float4& res, float new_weight, uchar4& cur, float& current_weight)
{
    uchar4 o;
    if (current_weight == 0) {
        o.x = (unsigned char)(res.x * 255.9999f);
        o.y = (unsigned char)(res.y * 255.9999f);
        o.z = (unsigned char)(res.z * 255.9999f);
        o.w = 255;
        current_weight = new_weight;
    } else {
        const float sum_wts = current_weight + new_weight;
        o.x = (unsigned char)__fdiv_rn(__fmaf_rn(__fmul_rn(res.x, new_weight), 255.9999f, __fmul_rn((float)cur.x, current_weight)), sum_wts);
        o.y = (unsigned char)__fdiv_rn(__fmaf_rn(__fmul_rn(res.y, new_weight), 255.9999f, __fmul_rn((float)cur.y, current_weight)), sum_wts);
        o.z = (unsigned char)__fdiv_rn(__fmaf_rn(__fmul_rn(res.z, new_weight), 255.9999f, __fmul_rn((float)cur.z, current_weight)), sum_wts);
        o.w = 255;
        current_weight = current_weight + new_weight;
    }
    cur = o;
}

// transform_and_blend (resample.cu:7-65)
__global__ void __launch_bounds__(256) blend_kernel(uchar4* __restrict__ canvas, int cw, int ch, cudaTextureObject_t frame, int fw, int fh,
                                                    int nw, int nh, const float* __restrict__ mat3x3, int tx, int ty,
                                                    cudaTextureObject_t mask, float* __restrict__ canvas_wts, cudaTextureObject_t frame_wts)
{
    __shared__ float t[9];
    if (threadIdx.x < 9) t[threadIdx.x] = mat3x3[threadIdx.x];
    __syncthreads();
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)nw * nh) return;
    const int y = (int)(i / nw), x = (int)(i - (long long)y * nw);
    const int pos_x = x + tx, pos_y = y + ty;
    if (pos_x < 0 || pos_x >= cw || pos_y < 0 || pos_y >= ch) return;
    float4 res;
    float new_weight;
    if (!blend_sample(x, y, t, fw, fh, frame, mask, frame_wts, res, new_weight)) return;
    const long long index = (long long)pos_y * cw + pos_x;
    float weight = canvas_wts[index];
    uchar4 pix = weight == 0 ? make_uchar4(0, 0, 0, 0) : canvas[index];
    blend_update(res, new_weight, pix, weight);
    canvas[index] = pix;
    canvas_wts[index] = weight;
}

// ---- mosaic of a frame stream --------------------------------------------------------------------------------

constexpr int kMosaicMaxFrames = 1024;      // frames per nm_mosaic_blend_bgra call (32 ballot words)
constexpr int kMosaicTileW = 64;            // canvas tile of one blend_stream_kernel CTA
constexpr int kMosaicTileH = 16;
constexpr int kMosaicRows = 4;              // canvas rows per thread
constexpr int kMosaicThreads = kMosaicTileW * kMosaicTileH / kMosaicRows;
static_assert(kMosaicTileW % 32 == 0 && kMosaicTileH % kMosaicRows == 0, "a warp covers 32 pixels of one row");

// N calls of transform_blend, frame after frame, in ONE pass over the canvas.  Within one transform_blend launch
// every canvas pixel is written by at most one thread ((x, y) -> (x + tx, y + ty) is injective), so N launches in
// order are, per pixel, the N updates in frame order -- which is what one thread here applies to its pixels held
// in registers.  The CTA finds the frames whose rect meets its tile with one ballot per 32 frames (ascending frame
// order = bit order), stages 32 frames' rects / matrices / textures at a time in shared memory, and walks the set
// bits.  Pixel (px, py) of frame k uses the local (px - tx, py - ty) the per-frame kernel gives it.
__global__ void __launch_bounds__(kMosaicThreads) blend_stream_kernel(uchar4* __restrict__ canvas, int cw, int ch, float* __restrict__ canvas_wts,
                                                                      const unsigned long long* __restrict__ frame_tex, int n,
                                                                      const float* __restrict__ mats, const int4* __restrict__ rects, int fw,
                                                                      int fh, cudaTextureObject_t mask, cudaTextureObject_t frame_wts)
{
    __shared__ unsigned s_hit[kMosaicMaxFrames / 32];
    __shared__ int4 s_rect[32];
    __shared__ float s_mat[32][9];
    __shared__ unsigned long long s_tex[32];
    const int x0 = blockIdx.x * kMosaicTileW, y0 = blockIdx.y * kMosaicTileH;
    const int x1 = min(x0 + kMosaicTileW, cw), y1 = min(y0 + kMosaicTileH, ch);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n_words = (n + 31) >> 5;
    bool any = false;
    for (int w = warp; w < n_words; w += kMosaicThreads / 32) {
        const int k = w * 32 + lane;
        bool hit = false;
        if (k < n) {
            const int4 r = rects[k];
            hit = r.z > 0 && r.w > 0 && r.x < x1 && (long long)r.x + r.z > x0 && r.y < y1 && (long long)r.y + r.w > y0;
        }
        const unsigned bits = __ballot_sync(0xffffffffu, hit);
        if (lane == 0) s_hit[w] = bits;
        any |= hit;
    }
    if (!__syncthreads_or(any)) return;

    const int px = x0 + threadIdx.x % kMosaicTileW;
    const int py0 = y0 + threadIdx.x / kMosaicTileW;
    constexpr int kRowStep = kMosaicThreads / kMosaicTileW;
    uchar4 pix[kMosaicRows];
    float wt[kMosaicRows];
    unsigned inside = 0, touched = 0;
#pragma unroll
    for (int j = 0; j < kMosaicRows; ++j) {
        const int py = py0 + j * kRowStep;
        pix[j] = make_uchar4(0, 0, 0, 0);
        wt[j] = 0.f;
        if (px < cw && py < ch) {
            const long long index = (long long)py * cw + px;
            pix[j] = canvas[index];
            wt[j] = canvas_wts[index];
            inside |= 1u << j;
        }
    }
    for (int w = 0; w < n_words; ++w) {
        unsigned bits = s_hit[w];
        if (!bits) continue;                                   // the same for every thread of the CTA
        if (threadIdx.x < 32 && ((bits >> threadIdx.x) & 1u)) {
            const int k = w * 32 + threadIdx.x;
            s_rect[threadIdx.x] = rects[k];
            s_tex[threadIdx.x] = frame_tex[k];
#pragma unroll
            for (int i = 0; i < 9; ++i) s_mat[threadIdx.x][i] = mats[(long long)k * 9 + i];
        }
        __syncthreads();
        while (bits) {
            const int b = __ffs(bits) - 1;
            bits &= bits - 1;
            const int4 r = s_rect[b];
            const long long lx = (long long)px - r.x;
            if (lx < 0 || lx >= r.z) continue;
            const cudaTextureObject_t tex = s_tex[b];
#pragma unroll
            for (int j = 0; j < kMosaicRows; ++j) {
                const long long ly = (long long)(py0 + j * kRowStep) - r.y;
                if (!((inside >> j) & 1u) || ly < 0 || ly >= r.w) continue;
                float4 res;
                float new_weight;
                if (blend_sample((int)lx, (int)ly, s_mat[b], fw, fh, tex, mask, frame_wts, res, new_weight)) {
                    blend_update(res, new_weight, pix[j], wt[j]);
                    touched |= 1u << j;
                }
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < kMosaicRows; ++j) {
        if (!((touched >> j) & 1u)) continue;
        const long long index = (long long)(py0 + j * kRowStep) * cw + px;
        canvas[index] = pix[j];
        canvas_wts[index] = wt[j];
    }
}

// Placement of a registered stream, fp64, row-major 3x3 (helpers in nm_chain.cuh).
constexpr int kPlaceThreads = 256;
constexpr int kPlaceBlock = 128;            // frames whose transforms are staged in shared memory at a time
constexpr double kPlaceMaxCoord = 1073741824.0;   // 2^30: footprints beyond this are not representable as rects

// One CTA.  G[k] = frame k -> mosaic: G[0] = anchor (identity if NULL), G[k+1] = G[k] . H[k]^-1, H[k] replaced by the
// identity (flag bit 0 of frame k+1) when status[k*3] == 0 or H[k] is singular / non-finite.  Footprint of frame k =
// the bounding box of its sampling box [-1, fw] x [-1, fh] mapped through G[k] (flag bit 1 and an empty rect when a
// corner has w <= 0, is non-finite or lies beyond 2^30).  G (n x 9 doubles) is both output and work space.
__global__ void __launch_bounds__(kPlaceThreads) place_kernel(const float* __restrict__ H, const int* __restrict__ status, int n, int fw, int fh,
                                                              const float* __restrict__ anchor, const int* __restrict__ origin, double* G,
                                                              float* __restrict__ mats, int4* rects, int* flags, int* __restrict__ bounds)
{
    __shared__ double s_g[kPlaceBlock][9];
    __shared__ int s_red[4][kPlaceThreads / 32];
    const int tid = threadIdx.x;
    // steps H[p]^-1 in parallel, written where G[p + 1] will go
    for (int p = tid; p < n - 1; p += kPlaceThreads) {
        double r[9];
        const bool ok = nm_chain_step(H + (long long)p * 9, status == nullptr || status[(long long)p * 3] != 0, r);
        for (int i = 0; i < 9; ++i) G[(long long)(p + 1) * 9 + i] = r[i];
        flags[p + 1] = ok ? 0 : 1;
    }
    if (tid == 0) flags[0] = 0;
    double g[9];                                               // thread 0: the running G
    for (int i = 0; i < 9; ++i) g[i] = anchor ? (double)anchor[i] : ((i % 4 == 0) ? 1.0 : 0.0);
    int mn_x = INT_MAX, mn_y = INT_MAX, mx_x = INT_MIN, mx_y = INT_MIN;   // over non-empty rects, max exclusive
    __syncthreads();
    for (int base = 0; base < n; base += kPlaceBlock) {
        const int cnt = min(kPlaceBlock, n - base);
        for (int i = tid; i < cnt * 9; i += kPlaceThreads) s_g[i / 9][i % 9] = G[(long long)base * 9 + i];
        __syncthreads();
        if (tid == 0) {
            for (int k = 0; k < cnt; ++k) {
                double nx[9];
                if (base + k == 0) {
                    for (int i = 0; i < 9; ++i) nx[i] = g[i];
                } else {
                    const double* s = s_g[k];
                    for (int r = 0; r < 3; ++r)
                        for (int c = 0; c < 3; ++c) nx[r * 3 + c] = g[r * 3] * s[c] + g[r * 3 + 1] * s[3 + c] + g[r * 3 + 2] * s[6 + c];
                }
                nm_renormalise(nx);
                for (int i = 0; i < 9; ++i) g[i] = s_g[k][i] = nx[i];
            }
        }
        __syncthreads();
        for (int i = tid; i < cnt * 9; i += kPlaceThreads) G[(long long)base * 9 + i] = s_g[i / 9][i % 9];
        if (tid < cnt) {
            const int k = base + tid;
            const double* a = s_g[tid];
            const double cx[4] = {-1.0, (double)fw, -1.0, (double)fw}, cy[4] = {-1.0, -1.0, (double)fh, (double)fh};
            double lo_x = INFINITY, lo_y = INFINITY, hi_x = -INFINITY, hi_y = -INFINITY;
            bool ok = true;
            for (int c = 0; c < 4; ++c) {
                const double w = a[6] * cx[c] + a[7] * cy[c] + a[8];
                const double u = (a[0] * cx[c] + a[1] * cy[c] + a[2]) / w, v = (a[3] * cx[c] + a[4] * cy[c] + a[5]) / w;
                ok = ok && w > 0.0 && fabs(u) <= kPlaceMaxCoord && fabs(v) <= kPlaceMaxCoord;   // false for NaN
                lo_x = fmin(lo_x, u); hi_x = fmax(hi_x, u); lo_y = fmin(lo_y, v); hi_y = fmax(hi_y, v);
            }
            int4 r = make_int4(0, 0, 0, 0);
            if (ok) {
                r.x = (int)floor(lo_x); r.y = (int)floor(lo_y);
                r.z = (int)ceil(hi_x) - r.x + 1; r.w = (int)ceil(hi_y) - r.y + 1;
                mn_x = min(mn_x, r.x); mn_y = min(mn_y, r.y); mx_x = max(mx_x, r.x + r.z); mx_y = max(mx_y, r.y + r.w);
            } else {
                flags[k] |= 2;
            }
            rects[k] = r;                                      // mosaic coordinates until the origin is known
        }
        __syncthreads();
    }
    // canvas origin and size: block reduction of the rect bounds
    const int lane = tid & 31, warp = tid >> 5;
    for (int o = 16; o; o >>= 1) {
        mn_x = min(mn_x, __shfl_xor_sync(0xffffffffu, mn_x, o)); mn_y = min(mn_y, __shfl_xor_sync(0xffffffffu, mn_y, o));
        mx_x = max(mx_x, __shfl_xor_sync(0xffffffffu, mx_x, o)); mx_y = max(mx_y, __shfl_xor_sync(0xffffffffu, mx_y, o));
    }
    if (lane == 0) { s_red[0][warp] = mn_x; s_red[1][warp] = mn_y; s_red[2][warp] = mx_x; s_red[3][warp] = mx_y; }
    __syncthreads();
    mn_x = INT_MAX; mn_y = INT_MAX; mx_x = INT_MIN; mx_y = INT_MIN;
    for (int i = 0; i < kPlaceThreads / 32; ++i) {
        mn_x = min(mn_x, s_red[0][i]); mn_y = min(mn_y, s_red[1][i]); mx_x = max(mx_x, s_red[2][i]); mx_y = max(mx_y, s_red[3][i]);
    }
    const bool none = mn_x > mx_x;                             // no frame has a footprint
    const int ox = origin ? origin[0] : (none ? 0 : mn_x), oy = origin ? origin[1] : (none ? 0 : mn_y);
    if (tid == 0) {
        bounds[0] = ox; bounds[1] = oy;
        bounds[2] = none ? 0 : max(0, mx_x - ox); bounds[3] = none ? 0 : max(0, mx_y - oy);
    }
    // per frame: rect relative to the origin, canvas-local -> frame matrix G^-1 . T(tx + ox, ty + oy)
    for (int k = tid; k < n; k += kPlaceThreads) {
        int4 r = rects[k];
        if (r.z == 0) r.x = r.y = 0; else { r.x -= ox; r.y -= oy; }
        rects[k] = r;
        double a[9], gi[9], m[9];
        for (int i = 0; i < 9; ++i) a[i] = G[(long long)k * 9 + i];
        nm_inv3d(a, nm_det3d(a), gi);
        const double sx = (double)r.x + ox, sy = (double)r.y + oy;
        for (int row = 0; row < 3; ++row) {
            m[row * 3] = gi[row * 3];
            m[row * 3 + 1] = gi[row * 3 + 1];
            m[row * 3 + 2] = gi[row * 3] * sx + gi[row * 3 + 1] * sy + gi[row * 3 + 2];
        }
        nm_renormalise(m);
        for (int i = 0; i < 9; ++i) mats[(long long)k * 9 + i] = (float)m[i];
    }
}

} // namespace

extern "C" int nm_resample_perspective_bgra(void* result, unsigned long long tex, int cols, int rows, float* x_pos, float* y_pos,
                                            const float* mat3x3, int inverse, nm_stream_t stream)
{
    if (cols < 0 || rows < 0) return NM_ERR_INVALID;
    const long long n = (long long)cols * rows;
    if (n == 0) return NM_OK;
    if (!result || !tex || !x_pos || !y_pos || !mat3x3) return NM_ERR_INVALID;
    const unsigned grid = (unsigned)nm_div_up64(n, 256);
    if (inverse)
        perspective_resample_kernel<true><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<uchar4*>(result), (cudaTextureObject_t)tex,
                                                                                  cols, rows, x_pos, y_pos, mat3x3);
    else
        perspective_resample_kernel<false><<<grid, 256, 0, (cudaStream_t)stream>>>(static_cast<uchar4*>(result), (cudaTextureObject_t)tex,
                                                                                   cols, rows, x_pos, y_pos, mat3x3);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_resample_mask_tex_u8(unsigned char* result, unsigned long long tex, int cols, int rows, const float* x_pos,
                                       const float* y_pos, float threshold, nm_stream_t stream)
{
    if (cols < 0 || rows < 0) return NM_ERR_INVALID;
    const long long n = (long long)cols * rows;
    if (n == 0) return NM_OK;
    if (!result || !tex || !x_pos || !y_pos) return NM_ERR_INVALID;
    resample_mask_kernel<<<(unsigned)nm_div_up64(n, 256), 256, 0, (cudaStream_t)stream>>>(result, (cudaTextureObject_t)tex, n, x_pos, y_pos,
                                                                                         threshold);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_transform_blend_bgra(void* canvas, int cw, int ch, unsigned long long frame_tex, int fw, int fh, int nw, int nh,
                                       const float* mat3x3, int tx, int ty, unsigned long long mask_tex, float* canvas_wts,
                                       unsigned long long frame_wts_tex, nm_stream_t stream)
{
    if (cw < 0 || ch < 0 || nw < 0 || nh < 0) return NM_ERR_INVALID;
    const long long n = (long long)nw * nh;
    if (n == 0 || (long long)cw * ch == 0) return NM_OK;
    if (!canvas || !frame_tex || !mat3x3 || !mask_tex || !canvas_wts || !frame_wts_tex) return NM_ERR_INVALID;
    blend_kernel<<<(unsigned)nm_div_up64(n, 256), 256, 0, (cudaStream_t)stream>>>(static_cast<uchar4*>(canvas), cw, ch,
                                                                                 (cudaTextureObject_t)frame_tex, fw, fh, nw, nh, mat3x3, tx, ty,
                                                                                 (cudaTextureObject_t)mask_tex, canvas_wts,
                                                                                 (cudaTextureObject_t)frame_wts_tex);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

// ---- mosaic of a frame stream: context, placement, blend -------------------------------------------------------

struct nm_mosaic_ctx {
    int fw = 0, fh = 0, max_frames = 0;
    std::vector<cudaArray_t> frame_arr;                        // one uchar4 array per frame slot
    std::vector<cudaTextureObject_t> frame_tex;
    unsigned long long* frame_tex_dev = nullptr;               // the same handles, for blend_stream_kernel
    cudaArray_t mask_arr = nullptr, wts_arr = nullptr;
    cudaTextureObject_t mask_tex = 0, wts_tex = 0;
};

namespace {
// the reference's CudaTex2D settings (gpu/utils/cudatex2D.cu:12-19): border addressing, linear filter, unnormalised
// coordinates
int make_texture(cudaArray_t arr, cudaTextureReadMode read_mode, cudaTextureObject_t* tex)
{
    cudaResourceDesc rd;
    std::memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = arr;
    cudaTextureDesc td;
    std::memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeBorder;
    td.filterMode = cudaFilterModeLinear;
    td.readMode = read_mode;
    td.normalizedCoords = 0;
    return nm_cuda_err(cudaCreateTextureObject(tex, &rd, &td, nullptr));
}

template <typename T>
int make_array(int w, int h, const void* init, cudaArray_t* arr)
{
    cudaChannelFormatDesc fd = cudaCreateChannelDesc<T>();
    cudaError_t e = cudaMallocArray(arr, &fd, w, h);
    if (e != cudaSuccess) { cudaGetLastError(); *arr = nullptr; return NM_ERR_ALLOC; }
    if (init) return nm_cuda_err(cudaMemcpy2DToArray(*arr, 0, 0, init, sizeof(T) * w, sizeof(T) * w, h, cudaMemcpyDefault));
    return NM_OK;
}
} // namespace

extern "C" int nm_mosaic_destroy(nm_mosaic_ctx* m)
{
    if (!m) return NM_OK;
    for (cudaTextureObject_t t : m->frame_tex) if (t) cudaDestroyTextureObject(t);
    for (cudaArray_t a : m->frame_arr) if (a) cudaFreeArray(a);
    if (m->mask_tex) cudaDestroyTextureObject(m->mask_tex);
    if (m->wts_tex) cudaDestroyTextureObject(m->wts_tex);
    if (m->mask_arr) cudaFreeArray(m->mask_arr);
    if (m->wts_arr) cudaFreeArray(m->wts_arr);
    if (m->frame_tex_dev) cudaFree(m->frame_tex_dev);
    delete m;
    return NM_OK;
}

extern "C" int nm_mosaic_create(nm_mosaic_ctx** out, int frame_w, int frame_h, int max_frames, const unsigned char* mask,
                                const float* weights)
{
    if (!out || !mask || !weights || frame_w <= 0 || frame_h <= 0 || max_frames <= 0 || max_frames > kMosaicMaxFrames)
        return NM_ERR_INVALID;
    *out = nullptr;
    const int cc = nm_device_cc();
    if (cc < 0) return cc;
    if (cc / 10 != 10) return NM_ERR_NO_DEVICE;
    nm_mosaic_ctx* m = new (std::nothrow) nm_mosaic_ctx();
    if (!m) return NM_ERR_ALLOC;
    m->fw = frame_w; m->fh = frame_h; m->max_frames = max_frames;
    m->frame_arr.assign(max_frames, nullptr);
    m->frame_tex.assign(max_frames, 0);
    int rc = make_array<unsigned char>(frame_w, frame_h, mask, &m->mask_arr);
    if (rc == NM_OK) rc = make_array<float>(frame_w, frame_h, weights, &m->wts_arr);
    if (rc == NM_OK) rc = make_texture(m->mask_arr, cudaReadModeNormalizedFloat, &m->mask_tex);
    if (rc == NM_OK) rc = make_texture(m->wts_arr, cudaReadModeElementType, &m->wts_tex);
    for (int i = 0; i < max_frames && rc == NM_OK; ++i) {
        rc = make_array<uchar4>(frame_w, frame_h, nullptr, &m->frame_arr[i]);
        if (rc == NM_OK) rc = make_texture(m->frame_arr[i], cudaReadModeNormalizedFloat, &m->frame_tex[i]);
    }
    if (rc == NM_OK && cudaMalloc(&m->frame_tex_dev, sizeof(unsigned long long) * max_frames) != cudaSuccess) {
        cudaGetLastError();
        m->frame_tex_dev = nullptr;
        rc = NM_ERR_ALLOC;
    }
    if (rc == NM_OK)
        rc = nm_cuda_err(cudaMemcpy(m->frame_tex_dev, m->frame_tex.data(), sizeof(unsigned long long) * max_frames, cudaMemcpyHostToDevice));
    if (rc != NM_OK) { nm_mosaic_destroy(m); return rc; }
    *out = m;
    return NM_OK;
}

extern "C" int nm_mosaic_textures(nm_mosaic_ctx* m, unsigned long long* frame_tex_host, unsigned long long* mask_tex,
                                  unsigned long long* wts_tex)
{
    if (!m) return NM_ERR_INVALID;
    if (frame_tex_host) for (int i = 0; i < m->max_frames; ++i) frame_tex_host[i] = m->frame_tex[i];
    if (mask_tex) *mask_tex = m->mask_tex;
    if (wts_tex) *wts_tex = m->wts_tex;
    return NM_OK;
}

extern "C" int nm_mosaic_place_f32(const float* H_pairs, const int* status, int n_frames, int frame_w, int frame_h,
                                   const float* anchor9, const int* origin2, float* mats_out, int* rects_out, int* flags_out,
                                   int* bounds_out, double* chain_out, nm_stream_t stream)
{
    if (n_frames <= 0 || frame_w <= 0 || frame_h <= 0 || (n_frames > 1 && !H_pairs) || !mats_out || !rects_out || !flags_out ||
        !bounds_out)
        return NM_ERR_INVALID;
    const cudaStream_t st = (cudaStream_t)stream;
    double* G = chain_out;
    if (!G) NM_CUDA_TRY(nm_ws_alloc(&G, sizeof(double) * 9 * (size_t)n_frames, st));
    place_kernel<<<1, kPlaceThreads, 0, st>>>(H_pairs, status, n_frames, frame_w, frame_h, anchor9, origin2, G, mats_out,
                                              reinterpret_cast<int4*>(rects_out), flags_out, bounds_out);
    const cudaError_t e = cudaGetLastError();
    if (!chain_out) cudaFreeAsync(G, st);
    return nm_cuda_err(e);
}

extern "C" int nm_mosaic_blend_bgra(nm_mosaic_ctx* m, const void* frames_bgra, int n_frames, int frame_w, int frame_h, const float* mats,
                                    const int* rects, void* canvas, int cw, int ch, float* canvas_wts, nm_stream_t stream)
{
    if (!m || !frames_bgra || !mats || !rects || !canvas || !canvas_wts || n_frames <= 0 || n_frames > m->max_frames || cw <= 0 ||
        ch <= 0 || frame_w != m->fw || frame_h != m->fh)
        return NM_ERR_INVALID;
    if (reinterpret_cast<uintptr_t>(rects) % 16 != 0) return NM_ERR_INVALID;
    const cudaStream_t st = (cudaStream_t)stream;
    const size_t row = sizeof(uchar4) * (size_t)m->fw;
    for (int i = 0; i < n_frames; ++i)
        NM_CUDA_TRY(cudaMemcpy2DToArrayAsync(m->frame_arr[i], 0, 0, static_cast<const unsigned char*>(frames_bgra) + row * m->fh * i, row, row,
                                             m->fh, cudaMemcpyDeviceToDevice, st));
    const dim3 grid((unsigned)nm_div_up(cw, kMosaicTileW), (unsigned)nm_div_up(ch, kMosaicTileH));
    if (grid.y > 65535) return NM_ERR_OVERFLOW;
    blend_stream_kernel<<<grid, kMosaicThreads, 0, st>>>(static_cast<uchar4*>(canvas), cw, ch, canvas_wts, m->frame_tex_dev, n_frames, mats,
                                                         reinterpret_cast<const int4*>(rects), m->fw, m->fh, m->mask_tex, m->wts_tex);
    NM_LAUNCH_CHECK();
    return NM_OK;
}
