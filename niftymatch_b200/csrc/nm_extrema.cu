// nm_extrema.cu -- DoG + 3x3x3 extrema + sub-pixel refinement + edge/contrast rejection
// + gradient maps, and the ordered compaction of the accepted keypoints.
//
// Replaces, for a whole batch and without host synchronisation:
//   compute_dog        (gpu/sift/siftfunctions.cu:42-51   -> 5x subtract, cudamath.cu:26)
//   compute_gradients  (gpu/sift/siftfunctions.cu:53-63   -> 3x gradient, cudamath.cu:38)
//   compute_keypoints  (gpu/sift/siftfunctions.cu:100-134 -> 5x cudaMallocArray + texture,
//                       3x thrust::fill + detect_keypoints, keypoint.cu:183-200)
//   PyramidData::gpu_collate_keypoints_for_level (gpu/sift/pyramidata.cu:84-91, copy_if)
//
// Design: the stencil pass (extrema_kernel) reads the 6 Gaussian levels of a tile once, forms
// the 5 DoG values in registers (never materialised in HBM), tests the 3 detection levels and
// lists the extremum candidates; refine_list_kernel refines/rejects them and sets ONE BIT per
// accepted pixel and level.  The ordered keypoint list ("copy_if order": raster within a
// level, levels ascending, octaves ascending) is then produced from the bitmaps: a per-segment
// popcount scan gives every word its rank, a tiny planning kernel applies the reference's
// early-return and capacity rules, an emit kernel writes each set bit's pixel at its final
// slot, and kprefine_kernel re-runs the (deterministic) refinement there and marks the
// gradient-map blocks the keypoint's windows read.  gradmap_kernel then computes only those
// blocks.  No dense float4 maps (16 B/pixel/level in the reference), no thrust::fill, no
// device->host count round trips.
#include "nm_sift_internal.cuh"
#include "nm_pyramid.cuh"
#include "nm_refine.cuh"
#include "nm_kpgeom.cuh"

namespace {

// 34 rows x 40 columns per level: tile column 0 sits at window column EX_HL = 4, because the innermost
// TMA coordinate has to stay 16-byte aligned (x0 - 4, not x0 - 1; unaligned starts raise an illegal-instruction fault)
constexpr int EX_TW = 32, EX_TH = 32, EX_HL = 4, EX_P = EX_TW + 2 * EX_HL, EX_ROWS = EX_TH + 2;
constexpr uint32_t EX_TILE_BYTES = 6u * EX_ROWS * EX_P * sizeof(float);   // 32 640

__device__ __forceinline__ uint32_t ex_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

struct GlobalDogFetch {
    const float* L;            // frame's level 0 at the candidate pixel
    long long le;              // level_elems
    int pitch, l;
    __device__ __forceinline__ float dogv(int k, int dx, int dy) const
    {
        const float* p = L + (long long)dy * pitch + dx;
        return __fsub_rn(__ldg(p + (k + 1) * le), __ldg(p + k * le));
    }
    __device__ __forceinline__ float cur(int dx, int dy) const { return dogv(l + 1, dx, dy); }
    __device__ __forceinline__ float down(int dx, int dy) const { return dogv(l, dx, dy); }
    __device__ __forceinline__ float up(int dx, int dy) const { return dogv(l + 2, dx, dy); }
};

// ------------------------- extrema and their refinement -------------------------
// DoG values formed on the fly from the staged Gaussian levels (cudamath.cu:34: next - this).
struct SmemLevelFetch {
    const float (*lv)[EX_ROWS][EX_P];      // [6]
    int l, r, c;                           // detection level (0..2), window row / column of the centre
    __device__ __forceinline__ float dogv(int k, int dx, int dy) const
    {
        return __fsub_rn(lv[k + 1][r + dy][c + dx], lv[k][r + dy][c + dx]);
    }
    __device__ __forceinline__ float cur(int dx, int dy) const { return dogv(l + 1, dx, dy); }
    __device__ __forceinline__ float down(int dx, int dy) const { return dogv(l, dx, dy); }
    __device__ __forceinline__ float up(int dx, int dy) const { return dogv(l + 2, dx, dy); }
};

constexpr int EX2_MAXC = EX_TW * EX_TH * 3;                     // every pixel of every level a candidate: cannot overflow
constexpr int EX2_LIST = 32;                                    // candidates of a tile handed to refine_list_kernel (one warp)
constexpr int EX2_SMEM = 2 * (int)EX_TILE_BYTES + EX2_MAXC * (int)sizeof(unsigned short) + 3 * EX_TH * 4 + 64;   // 71 872: 3 CTAs / SM

// Persistent CTAs walk the 32 x 32 tiles of a launch (x fastest, so the CTAs in flight work on neighbouring
// tiles and the halo columns / rows they share are L2 hits).  The six-level window of the NEXT tile is
// fetched by TMA into the other half of a double buffer while the current one is processed: the window is
// read-only (the DoG differences are formed in registers), so no thread waits for a load at CTA start
// (13.8 % of the stall samples of the fused round-1 kernel) and the DoG pass with its barrier is gone.
// Per tile: the separable 26-neighbour test for 4 pixels x 3 levels per thread, the Gaussian levels carried
// in registers from one DoG level to the next; the extremum candidates (about 0.2 % of the pixels) go to a
// list in shared memory and, after the tile's ONE barrier, to the tile's slot of a global list that
// refine_list_kernel works through with one lane per candidate -- in this kernel the ~300-instruction
// refinement (IEEE divisions, a dependent chain of ~1500 cycles) would leave seven warps waiting at a barrier
// for the one that has a candidate.  Tiles with more than 32 candidates (not seen on images; possible on
// synthetic noise) are refined here.  Gradient maps are not produced here (gradmap_kernel).
__global__ void __launch_bounds__(256, 3) extrema_kernel(const NmOctave oc, const NmDetectParams dp,
                                                         const __grid_constant__ CUtensorMap tmap,
                                                         int tiles_x, int tiles_y, int n_tiles,
                                                         int* __restrict__ cand_n, unsigned short* __restrict__ cand)
{
    extern __shared__ __align__(128) unsigned char ex_smem[];
    float (*s_win)[6][EX_ROWS][EX_P] = reinterpret_cast<float (*)[6][EX_ROWS][EX_P]>(ex_smem);      // [2]
    unsigned short* s_cand = reinterpret_cast<unsigned short*>(ex_smem + 2 * EX_TILE_BYTES);                               // [EX2_MAXC], read by crowded tiles only
    unsigned (*s_bits)[EX_TH] = reinterpret_cast<unsigned (*)[EX_TH]>(ex_smem + 2 * EX_TILE_BYTES + EX2_MAXC * 2);        // [3], crowded tiles only
    uint64_t* s_bar = reinterpret_cast<uint64_t*>(ex_smem + 2 * EX_TILE_BYTES + EX2_MAXC * 2 + 3 * EX_TH * 4);             // [2]
    // candidate counters rotate over three slots: slot it % 3 is pushed to before tile it's barrier, read after it, and
    // cleared after the barrier of tile it + 1 (every thread has read it by then; the next pushes come after barrier it + 2)
    int* s_ncand = reinterpret_cast<int*>(s_bar + 2);                                                                      // [3]
    const int tid = threadIdx.y * 32 + threadIdx.x, lane = threadIdx.x;
    const long long bm_words = (long long)oc.h * oc.wpr;
    const int nrb = (oc.h + NM_NEED_ROWS - 1) / NM_NEED_ROWS;

    auto issue = [&](int tile, int buf) {
        const int tx = tile % tiles_x, q = tile / tiles_x, ty = q % tiles_y, f = q / tiles_y;
        const uint32_t bar = ex_smem_u32(&s_bar[buf]);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(EX_TILE_BYTES) : "memory");
        asm volatile(
            "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
            ::"r"(ex_smem_u32(&s_win[buf][0][0][0])), "l"(reinterpret_cast<uint64_t>(&tmap)), "r"(tx * EX_TW - EX_HL),
              "r"(ty * EX_TH - 1), "r"(f * 6), "r"(bar) : "memory");
    };

    int tile = blockIdx.x;
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ex_smem_u32(&s_bar[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(ex_smem_u32(&s_bar[1])));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        s_ncand[0] = s_ncand[1] = s_ncand[2] = 0;
        if (tile < n_tiles) issue(tile, 0);
    }
    __syncthreads();

    const float t = __fmul_rn(0.8f, dp.peak);
    for (int it = 0; tile < n_tiles; ++it, tile += gridDim.x) {
        const int buf = it & 1, cnt = it % 3;
        const int tx = tile % tiles_x, q = tile / tiles_x, ty = q % tiles_y, f = q / tiles_y;
        const int x0 = tx * EX_TW, y0 = ty * EX_TH;
        // the other buffer was last read before the barrier of the previous iteration
        if (tid == 0 && tile + (int)gridDim.x < n_tiles) issue(tile + gridDim.x, buf ^ 1);
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "LAB_WAIT_%=:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra LAB_DONE_%=;\n"
            "bra LAB_WAIT_%=;\n"
            "LAB_DONE_%=:\n"
            "}\n" ::"r"(ex_smem_u32(&s_bar[buf])), "r"((it >> 1) & 1) : "memory");
        const float (*L)[EX_ROWS][EX_P] = s_win[buf];

        // ---- separable 26-neighbour test, same comparisons as keypoint.cu:19-105 / :195-196 ----
        unsigned extmask = 0;                      // bit l * 4 + j
        {
            const int c = lane + EX_HL, rbase = threadIdx.y * (EX_TH / 8);     // window row of the first pixel's upper neighbour
            float lo[6][3];                        // Gaussian level k at the thread's 6 rows x 3 columns
#pragma unroll
            for (int rr = 0; rr < 6; ++rr) {
                lo[rr][0] = L[0][rbase + rr][c - 1]; lo[rr][1] = L[0][rbase + rr][c]; lo[rr][2] = L[0][rbase + rr][c + 1];
            }
            float m9x[3][4], m9n[3][4];            // ring over k % 3: 3x3 maxima / minima, centre included
            float m8x[4], m8n[4], cv[4];           // DoG level k - 1 (centre excluded) and its centre values
            float p8x[4], p8n[4], pcv[4];
#pragma unroll
            for (int k = 0; k < 5; ++k) {
                float hx[6], hn[6], gxm[6], gnm[6], ctr[6];
#pragma unroll
                for (int rr = 0; rr < 6; ++rr) {
                    const float u0 = L[k + 1][rbase + rr][c - 1], u1 = L[k + 1][rbase + rr][c], u2 = L[k + 1][rbase + rr][c + 1];
                    const float a = __fsub_rn(u0, lo[rr][0]), b = __fsub_rn(u1, lo[rr][1]), d = __fsub_rn(u2, lo[rr][2]);
                    lo[rr][0] = u0; lo[rr][1] = u1; lo[rr][2] = u2;
                    hx[rr] = fmaxf(fmaxf(a, b), d);
                    hn[rr] = fminf(fminf(a, b), d);
                    gxm[rr] = fmaxf(a, d);
                    gnm[rr] = fminf(a, d);
                    ctr[rr] = b;
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    m9x[k % 3][j] = fmaxf(fmaxf(hx[j], hx[j + 1]), hx[j + 2]);
                    m9n[k % 3][j] = fminf(fminf(hn[j], hn[j + 1]), hn[j + 2]);
                    p8x[j] = m8x[j]; p8n[j] = m8n[j]; pcv[j] = cv[j];
                    m8x[j] = fmaxf(fmaxf(hx[j], gxm[j + 1]), hx[j + 2]);
                    m8n[j] = fminf(fminf(hn[j], gnm[j + 1]), hn[j + 2]);
                    cv[j] = ctr[j + 1];
                }
                if (k >= 2) {
                    const int l = k - 2;
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const float mx = fmaxf(fmaxf(m9x[(k - 2) % 3][j], p8x[j]), m9x[k % 3][j]);
                        const float mn = fminf(fminf(m9n[(k - 2) % 3][j], p8n[j]), m9n[k % 3][j]);
                        const float c0 = pcv[j];
                        if ((c0 <= t && c0 < mn) || (c0 >= t && c0 > mx)) extmask |= 1u << (l * 4 + j);
                    }
                }
            }
            // interior pixels only (keypoint.cu:191)
            const int gx = x0 + lane;
            if (!(gx >= 1 && gx <= oc.w - 2)) extmask = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int gy = y0 + rbase + j;
                if (!(gy >= 1 && gy <= oc.h - 2)) extmask &= ~(0x111u << j);
            }
        }
        if (extmask) {
            const int n = __popc(extmask);
            int pos = atomicAdd(&s_ncand[cnt], n);
            while (extmask) {
                const int b = __ffs(extmask) - 1;
                extmask &= extmask - 1;
                // level (2 bits) | tile row (5 bits) | tile column (5 bits); the first EX2_LIST straight to the tile's global list
                const unsigned short e = (unsigned short)(((b >> 2) << 10) | ((threadIdx.y * (EX_TH / 8) + (b & 3)) << 5) | lane);
                s_cand[pos] = e;
                if (pos < EX2_LIST) cand[(long long)tile * EX2_LIST + pos] = e;
                ++pos;
            }
        }
        __syncthreads();

        const int ncand = s_ncand[cnt];
        // the tile's bitmap words and its blocks of the gradient-need map start clear (set by refine_list_kernel /
        // below, marked by kprefine_kernel)
        if (tid < 3 * EX_TH) {
            const int l = tid / EX_TH, gy = y0 + tid % EX_TH;
            if (gy < oc.h) oc.bitmap[((long long)f * 3 + l) * bm_words + (long long)gy * oc.wpr + tx] = 0u;
        } else if (tid < 3 * EX_TH + 3 * (EX_TH / NM_NEED_ROWS)) {
            const int i = tid - 3 * EX_TH;
            const int l = i / (EX_TH / NM_NEED_ROWS), rb = ty * (EX_TH / NM_NEED_ROWS) + i % (EX_TH / NM_NEED_ROWS);
            if (rb < nrb) oc.need[(((long long)f * 3 + l) * nrb + rb) * oc.wpr + tx] = 0;
        } else if (tid == 255) {
            cand_n[tile] = ncand <= EX2_LIST ? ncand : 0;
            s_ncand[(it + 2) % 3] = 0;             // the previous tile's counter
        }
        if (ncand > EX2_LIST) {
            // ---- crowded tile: refined here (keypoint.cu:108-180, 214), bits through shared memory ----
            if (tid < 3 * EX_TH) (&s_bits[0][0])[tid] = 0u;
            __syncthreads();
            for (int i = tid; i < ncand; i += 256) {
                const unsigned e = s_cand[i];
                const int l = e >> 10, ly = (e >> 5) & 31, lx = e & 31;
                const int gx = x0 + lx, gy = y0 + ly;
                const bool masked_out = dp.mask != 0 &&
                    tex2D<float>((cudaTextureObject_t)dp.mask, (gx + 0.5f) * oc.xper, (gy + 0.5f) * oc.xper) < 1.f;
                if (!masked_out) {
                    SmemLevelFetch ft{L, l, ly + 1, lx + EX_HL};
                    float4 out;
                    if (nm_refine(ft, gx, gy, dp.peak, dp.edge, oc.xper, dp.sigma_0, dp.num_dogs, l, out))
                        atomicOr(&s_bits[l][ly], 1u << lx);
                }
            }
            __syncthreads();
            if (tid < 3 * EX_TH) {
                const int l = tid / EX_TH, ly = tid % EX_TH, gy = y0 + ly;
                if (gy < oc.h) oc.bitmap[((long long)f * 3 + l) * bm_words + (long long)gy * oc.wpr + tx] = s_bits[l][ly];
            }
            __syncthreads();                       // s_cand / the window are rewritten by the next tiles
        }
    }
}

// One warp per tile of the extrema launch, one lane per listed candidate: mask test (keypoint.cu:214), refinement
// and rejection (keypoint.cu:108-180) on DoG values formed from the Gaussian levels in global memory (L2 hits: the
// extrema kernel has just read them); accepted pixels set their bit in the keypoint bitmap.
__global__ void __launch_bounds__(256) refine_list_kernel(const NmOctave oc, const NmDetectParams dp, int tiles_x, int tiles_y,
                                                          int n_tiles, const int* __restrict__ cand_n,
                                                          const unsigned short* __restrict__ cand)
{
    const int tile = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (tile >= n_tiles) return;
    if (lane >= cand_n[tile]) return;
    const unsigned e = cand[(long long)tile * EX2_LIST + lane];
    const int tx = tile % tiles_x, q = tile / tiles_x, ty = q % tiles_y, f = q / tiles_y;
    const int l = e >> 10, gy = ty * EX_TH + ((e >> 5) & 31), gx = tx * EX_TW + (e & 31);
    if (dp.mask != 0 && tex2D<float>((cudaTextureObject_t)dp.mask, (gx + 0.5f) * oc.xper, (gy + 0.5f) * oc.xper) < 1.f) return;
    GlobalDogFetch ft{oc.levels + (long long)f * 6 * oc.level_elems + (long long)gy * oc.pitch + gx, oc.level_elems, oc.pitch, l};
    float4 out;
    if (nm_refine(ft, gx, gy, dp.peak, dp.edge, oc.xper, dp.sigma_0, dp.num_dogs, l, out))
        atomicOr(oc.bitmap + ((long long)f * 3 + l) * oc.h * oc.wpr + (long long)gy * oc.wpr + tx, 1u << (e & 31));
}

// Gradient maps of levels 1..3 (compute_gradients, siftfunctions.cu:53-63 -> cudamath.cu:38-54; border
// pixels = (0, 0)), restricted to the 8-row x 32-column blocks that an orientation or descriptor window
// touches (need map, marked by kprefine_kernel).  A CTA covers 256 columns x 32 rows of one level: a warp
// owns a 32-column strip and walks its four blocks; lane = column.  The four neighbours come straight from
// global memory (the rows are L1 / L2 hits of the neighbouring lanes and rows), all 26 loads of a block in
// flight before its first gradient is evaluated.  `dense` != 0 computes every block (tests and tools that read
// whole maps).
// R interior rows of a gradient map starting at `p0` (the source pixel of the first row) / `q` (its gradient): no
// per-row predicates, all loads first, all R gradients through the branch-free main path (their chains interleave),
// exact zeros (flat image areas) selected, the rare out-of-range arguments repaired afterwards.
template <int R>
__device__ __forceinline__ void gradmap_rows(const float* __restrict__ p0, float2* __restrict__ q, int pitch, bool intx)
{
    float ctr[R + 2], lf[R], rt[R];
    const float* __restrict__ p = p0 - pitch;
    ctr[0] = __ldg(p);
#pragma unroll
    for (int j = 0; j < R; ++j) {
        p += pitch;
        lf[j] = __ldg(p - 1); ctr[j + 1] = __ldg(p); rt[j] = __ldg(p + 1);
    }
    ctr[R + 1] = __ldg(p + pitch);
    float2 g[R];
    unsigned bad = 0;
#pragma unroll
    for (int j = 0; j < R; ++j) {
        const float dx = __fsub_rn(rt[j], lf[j]), dy = __fsub_rn(ctr[j + 2], ctr[j]);
        g[j] = nm_gradient_main(dx, dy);
        const bool zero = dx == 0.f && dy == 0.f;                   // library result: (0, 0)
        if (zero || !intx) g[j] = make_float2(0.f, 0.f);
        if (!zero && intx && !nm_gradient_in_range(dx, dy)) bad |= 1u << j;
    }
    if (bad) {
#pragma unroll
        for (int j = 0; j < R; ++j)
            if ((bad >> j) & 1u) g[j] = nm_gradient_lib(__fsub_rn(rt[j], lf[j]), __fsub_rn(ctr[j + 2], ctr[j]));
    }
#pragma unroll
    for (int j = 0; j < R; ++j) {
        *q = g[j];
        q += pitch;
    }
}

// What was measured on 64 x 1080p frames (ms for the stage): 72 registers / 3 CTAs per SM 1.49; this version (64
// registers, 4 CTAs) 1.32; 4- and 2-row sub-blocks at 5 - 8 CTAs (spilling) 1.34 - 1.53; prefetching the next block's
// loads (117 registers, 2 CTAs) 1.87; TMA-staged 32 x 32 tiles in persistent CTAs (the layout of extrema_kernel) 1.57.
// The kernel waits on its global loads (long-scoreboard 32 % of the stall samples): resident warps are what it needs.
__global__ void __launch_bounds__(256, 4) gradmap_kernel(const NmOctave oc, int strips_x, int dense)
{
    const int lane = threadIdx.x & 31;
    const int cb = (blockIdx.x % strips_x) * 8 + (threadIdx.x >> 5), rb0 = (blockIdx.x / strips_x) * 4;
    const int fl = blockIdx.y;                                  // frame * 3 + level
    const int w = oc.w, h = oc.h, pitch = oc.pitch, wpr = oc.wpr;
    const int x = cb * 32 + lane;
    if (cb >= wpr || x >= w) return;
    const int nrb = (h + NM_NEED_ROWS - 1) / NM_NEED_ROWS;
    const int f = fl / 3, l = fl - 3 * f;
    const unsigned char* __restrict__ need = oc.need + ((long long)fl * nrb) * wpr + cb;
    const float* __restrict__ src = oc.levels + ((long long)f * 6 + l + 1) * oc.level_elems + x;
    float2* __restrict__ G = oc.grad + (long long)fl * oc.level_elems + x;
    const bool intx = x >= 1 && x <= w - 2;
#pragma unroll 1
    for (int k = 0; k < 4; ++k) {
        const int rb = rb0 + k;
        if (rb >= nrb) break;
        if (!dense && need[rb * wpr] == 0) continue;            // warp uniform
        const int y0 = rb * NM_NEED_ROWS;
        if (y0 >= 1 && y0 + NM_NEED_ROWS + 1 <= h) {
            // rows y0 - 1 .. y0 + 8 exist (all but the first and last row block of a level): nothing is predicated per row.
            // The +-1 column neighbours of the first / last column read a pad element or the neighbouring row (inside
            // the level's allocation; unused: those lanes store (0, 0)).
            gradmap_rows<NM_NEED_ROWS>(src + (long long)y0 * pitch, G + (long long)y0 * pitch, pitch, intx);
            continue;
        }
        const float* __restrict__ p = src + (long long)y0 * pitch;
        float2* __restrict__ q = G + (long long)y0 * pitch;
        float ctr[NM_NEED_ROWS + 2], lf[NM_NEED_ROWS], rt[NM_NEED_ROWS];
#pragma unroll
        for (int j = -1; j <= NM_NEED_ROWS; ++j) {
            const int y = y0 + j;
            ctr[j + 1] = (intx && y >= 0 && y < h) ? __ldg(p + j * pitch) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < NM_NEED_ROWS; ++j) {
            const int y = y0 + j;
            const bool interior = intx && y >= 1 && y <= h - 2;
            lf[j] = interior ? __ldg(p + j * pitch - 1) : 0.f;
            rt[j] = interior ? __ldg(p + j * pitch + 1) : 0.f;
        }
#pragma unroll
        for (int j = 0; j < NM_NEED_ROWS; ++j) {
            const int y = y0 + j;
            if (y < h) {
                const bool interior = intx && y >= 1 && y <= h - 2;
                float2 g = make_float2(0.f, 0.f);
                if (interior) g = nm_gradient_at(rt[j], lf[j], ctr[j + 2], ctr[j]);
                q[j * pitch] = g;
            }
        }
    }
}

// One block per (segment, frame): exclusive prefix of the word popcounts + segment total.
// Coalesced: the block walks the bitmap in spans of 1024 words (4 consecutive words per thread, one
// 16-byte load), scans the span with warp shuffles, and carries the running total across spans.
__global__ void __launch_bounds__(256) rank_kernel(const NmOctaveTable tab, int* __restrict__ seg_raw)
{
    __shared__ int s_warp[8];
    __shared__ int s_carry;
    const int s = blockIdx.x, f = blockIdx.y, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const NmOctave& oc = tab.o[s / 3];
    const int l = s % 3;
    const int nwords = oc.h * oc.wpr;
    const uint32_t* __restrict__ bm = oc.bitmap + ((long long)f * 3 + l) * nwords;
    int* __restrict__ wp = oc.wprefix + ((long long)f * 3 + l) * nwords;
    const bool vec = ((reinterpret_cast<uintptr_t>(bm) | reinterpret_cast<uintptr_t>(wp)) & 15) == 0;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base < nwords; base += 1024) {
        const int i0 = base + tid * 4;
        uint4 w = make_uint4(0u, 0u, 0u, 0u);
        if (vec && i0 + 3 < nwords) {
            w = *reinterpret_cast<const uint4*>(bm + i0);
        } else {
            if (i0 < nwords) w.x = bm[i0];
            if (i0 + 1 < nwords) w.y = bm[i0 + 1];
            if (i0 + 2 < nwords) w.z = bm[i0 + 2];
            if (i0 + 3 < nwords) w.w = bm[i0 + 3];
        }
        const int c0 = __popc(w.x), c1 = __popc(w.y), c2 = __popc(w.z), c3 = __popc(w.w);
        const int mine = c0 + c1 + c2 + c3;
        int incl = mine;                                   // inclusive scan over the warp
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, d);
            if (lane >= d) incl += v;
        }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        int off = s_carry;
        for (int k = 0; k < wid; ++k) off += s_warp[k];
        const int e0 = off + incl - mine;
        if (vec && i0 + 3 < nwords) {
            *reinterpret_cast<int4*>(wp + i0) = make_int4(e0, e0 + c0, e0 + c0 + c1, e0 + c0 + c1 + c2);
        } else {
            if (i0 < nwords) wp[i0] = e0;
            if (i0 + 1 < nwords) wp[i0 + 1] = e0 + c0;
            if (i0 + 2 < nwords) wp[i0 + 2] = e0 + c0 + c1;
            if (i0 + 3 < nwords) wp[i0 + 3] = e0 + c0 + c1 + c2;
        }
        __syncthreads();
        if (tid == 255) s_carry = off + incl;
        __syncthreads();
    }
    if (tid == 0) seg_raw[f * tab.n_oct * 3 + s] = s_carry;
}

// Early-return rule (siftfunctions.cu:145,160: the first empty level ends the octave),
// output offsets in (octave, level) order, capacity truncation (siftfunctions.cu:166-169).
__global__ void plan_kernel(const int* __restrict__ seg_raw, int* __restrict__ seg_cnt,
                            int* __restrict__ seg_off, int* __restrict__ counts, int n_oct, int batch,
                            int capacity)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= batch) return;
    const int S = n_oct * 3;
    int off = 0;
    for (int o = 0; o < n_oct; ++o) {
        bool stopped = false;
        for (int l = 0; l < 3; ++l) {
            int c = seg_raw[f * S + o * 3 + l];
            if (stopped) c = 0;
            if (c == 0) stopped = true;
            seg_cnt[f * S + o * 3 + l] = c;
            seg_off[f * S + o * 3 + l] = off;
            off += c;
        }
    }
    counts[f] = off < capacity ? off : capacity;
}


// The blocks of the level's gradient map that the keypoint's orientation window (orientation.cu:43-53) and
// descriptor window (descriptor.cu:57-65, diagonal 16 x 16 chunks :94-97) read: same geometry routines as
// orient_kernel / describe_kernel (nm_kpgeom.cuh), so the marked set is a superset of the samples.
__device__ __forceinline__ void mark_rect(unsigned char* need, int wpr, int x0, int x1, int y0, int y1)
{
    if (x0 > x1 || y0 > y1) return;
    for (int rb = y0 / NM_NEED_ROWS; rb <= y1 / NM_NEED_ROWS; ++rb)
        for (int cb = x0 >> 5; cb <= (x1 >> 5); ++cb) need[(long long)rb * wpr + cb] = 1;
}
__device__ __forceinline__ void mark_gradient_need(const NmOctave& oc, int f, const float4 kp)
{
    const KpGeom g = kp_geom(kp, oc.xper);
    if (g.level < 0 || g.level > 2) return;
    const int nrb = (oc.h + NM_NEED_ROWS - 1) / NM_NEED_ROWS;
    unsigned char* need = oc.need + ((long long)f * 3 + g.level) * nrb * oc.wpr;
    float sigma_w;
    const int W = kp_orient_radius(g, sigma_w);
    mark_rect(need, oc.wpr, g.xi + max(-W, -g.xi), g.xi + min(W, oc.w - 1 - g.xi),
              g.yi + max(-W, -g.yi), g.yi + min(W, oc.h - 1 - g.yi));
    if (g.xi < 0 || g.xi >= oc.w || g.yi < 0 || g.yi >= oc.h) return;     // descriptor.cu:49
    const KpDescWindow d = kp_desc_window(g, oc.w, oc.h);
    for (int c = 0; c < d.chunks; ++c)
        mark_rect(need, oc.wpr, g.xi + d.xmin + 16 * c, g.xi + min(d.xmin + 16 * c + 15, d.xmax),
                  g.yi + d.ymin + 16 * c, g.yi + min(d.ymin + 16 * c + 15, d.ymax));
}

// Ordered compaction, step 3: every set bit of the bitmaps gets its slot (segment offset + word prefix + bits
// below it = copy_if order) and the slot receives the pixel (x, y, level) as integers.  One thread per word.
__global__ void __launch_bounds__(256) emit_kernel(const NmOctave oc, int octave_index, int n_oct,
                                                   const int* __restrict__ seg_cnt,
                                                   const int* __restrict__ seg_off, int capacity,
                                                   float4* __restrict__ kpts, int* __restrict__ meta)
{
    const int wi = blockIdx.x * 256 + threadIdx.x, l = blockIdx.y, f = blockIdx.z;
    const int nwords = oc.h * oc.wpr;
    if (wi >= nwords) return;
    const int S = n_oct * 3, s = octave_index * 3 + l;
    if (seg_cnt[f * S + s] == 0) return;
    uint32_t bits = oc.bitmap[((long long)f * 3 + l) * nwords + wi];
    if (!bits) return;
    int pos = seg_off[f * S + s] + oc.wprefix[((long long)f * 3 + l) * nwords + wi];
    const int y = wi / oc.wpr, xw = wi - y * oc.wpr;
    while (bits) {
        const int b = __ffs(bits) - 1;
        bits &= bits - 1;
        if (pos >= capacity) break;
        kpts[(long long)f * capacity + pos] = make_float4(__int_as_float(xw * 32 + b), __int_as_float(y), __int_as_float(l), -1.f);
        meta[(long long)f * capacity + pos] = octave_index;
        ++pos;
    }
}

// Step 4: one thread per emitted keypoint re-runs the (deterministic) refinement of its pixel from the Gaussian
// levels and writes the float4 payload (keypoint.cu:172-175) over the slot; it also marks the blocks of the
// gradient maps that the keypoint's windows read.  Dense threads: a warp refines 32 keypoints, where the
// per-word kernel above would run the ~400-instruction refinement (double pow) with one live lane.
__global__ void __launch_bounds__(256) kprefine_kernel(const NmOctaveTable tab, const NmDetectParams dp, int capacity,
                                                       const int* __restrict__ counts, float4* __restrict__ kpts,
                                                       const int* __restrict__ meta)
{
    const int j = blockIdx.x * 256 + threadIdx.x, f = blockIdx.y;
    if (j >= counts[f]) return;
    const long long kidx = (long long)f * capacity + j;
    const float4 slot = kpts[kidx];
    const int x = __float_as_int(slot.x), y = __float_as_int(slot.y), l = __float_as_int(slot.z);
    const NmOctave& oc = tab.o[meta[kidx]];
    GlobalDogFetch ft{oc.levels + (long long)f * 6 * oc.level_elems + (long long)y * oc.pitch + x, oc.level_elems, oc.pitch, l};
    float4 out = make_float4(-1.f, -1.f, -1.f, -1.f);
    nm_refine(ft, x, y, dp.peak, dp.edge, oc.xper, dp.sigma_0, dp.num_dogs, l, out);
    kpts[kidx] = out;
    if (out.w >= 0.f) mark_gradient_need(oc, f, out);
}

// ------------------------- compat: dense per-pixel maps -------------------------
struct LinearDogFetch {
    const float *c, *d, *u;    // at the candidate pixel
    int w;
    __device__ __forceinline__ float cur(int dx, int dy) const { return __ldg(c + dy * w + dx); }
    __device__ __forceinline__ float down(int dx, int dy) const { return __ldg(d + dy * w + dx); }
    __device__ __forceinline__ float up(int dx, int dy) const { return __ldg(u + dy * w + dx); }
};

__global__ void keypoints_dense_linear_kernel(const float* __restrict__ cur, const float* __restrict__ down,
                                              const float* __restrict__ up, cudaTextureObject_t mask, int w, int h,
                                              NmDetectParams dp, float xper, int level, float4* __restrict__ result)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < 1 || x > w - 2 || y < 1 || y > h - 2) return;       // keypoint.cu:191
    if (mask != 0 && tex2D<float>(mask, (x + 0.5f) * xper, (y + 0.5f) * xper) < 1.f) return;   // keypoint.cu:214
    const long long i = (long long)y * w + x;
    LinearDogFetch ft{cur + i, down + i, up + i, w};
    if (!nm_is_extremum(ft, dp.peak)) return;
    float4 out;
    if (nm_refine(ft, x, y, dp.peak, dp.edge, xper, dp.sigma_0, dp.num_dogs, level, out)) result[i] = out;
}

struct TexDogFetch {
    cudaTextureObject_t c, d, u;
    float ax, ay;
    __device__ __forceinline__ float cur(int dx, int dy) const { return tex2D<float>(c, ax + dx, ay + dy); }
    __device__ __forceinline__ float down(int dx, int dy) const { return tex2D<float>(d, ax + dx, ay + dy); }
    __device__ __forceinline__ float up(int dx, int dy) const { return tex2D<float>(u, ax + dx, ay + dy); }
};

__global__ void keypoints_dense_tex_kernel(cudaTextureObject_t cur, cudaTextureObject_t mask,
                                           cudaTextureObject_t down, cudaTextureObject_t up, int w, int h,
                                           NmDetectParams dp, float xper, int level, float4* __restrict__ result)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < 1 || x > w - 2 || y < 1 || y > h - 2) return;
    // keypoint.cu:214
    if (mask != 0 && tex2D<float>(mask, (x + 0.5f) * xper, (y + 0.5f) * xper) < 1.f) return;
    TexDogFetch ft{cur, down, up, x + 0.5f, y + 0.5f};
    if (!nm_is_extremum(ft, dp.peak)) return;
    float4 out;
    if (nm_refine(ft, x, y, dp.peak, dp.edge, xper, dp.sigma_0, dp.num_dogs, level, out))
        result[(long long)y * w + x] = out;
}

// ------------------------- compat: ordered copy_if ------------------------------
constexpr int COL_CHUNK = 2048;     // pixels per block
__global__ void __launch_bounds__(256) collate_count_kernel(const float4* __restrict__ dense, int n,
                                                            int* __restrict__ block_counts)
{
    __shared__ int s_cnt;
    if (threadIdx.x == 0) s_cnt = 0;
    __syncthreads();
    const int base = blockIdx.x * COL_CHUNK;
    int c = 0;
    for (int i = threadIdx.x; i < COL_CHUNK; i += 256) {
        const int p = base + i;
        if (p < n && dense[p].w >= 0.f) ++c;                    // pyramidata.cu:13
    }
    atomicAdd(&s_cnt, c);
    __syncthreads();
    if (threadIdx.x == 0) block_counts[blockIdx.x] = s_cnt;
}
__global__ void collate_scan_kernel(int* __restrict__ block_counts, int nblocks, int* __restrict__ total)
{
    // single thread: nblocks is small (n / 2048)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        int run = 0;
        for (int i = 0; i < nblocks; ++i) { int c = block_counts[i]; block_counts[i] = run; run += c; }
        *total = run;
    }
}
__global__ void __launch_bounds__(256) collate_write_kernel(const float4* __restrict__ dense, int n,
                                                            const int* __restrict__ block_offsets,
                                                            float4* __restrict__ out)
{
    __shared__ int s_warp[8];
    __shared__ int s_run;
    const int base = blockIdx.x * COL_CHUNK;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) s_run = block_offsets[blockIdx.x];
    __syncthreads();
    for (int i0 = 0; i0 < COL_CHUNK; i0 += 256) {
        const int p = base + i0 + threadIdx.x;
        float4 v = make_float4(-1.f, -1.f, -1.f, -1.f);
        if (p < n) v = dense[p];
        const bool keep = p < n && v.w >= 0.f;
        const unsigned m = __ballot_sync(0xffffffffu, keep);
        if (lane == 0) s_warp[wid] = __popc(m);
        __syncthreads();
        int off = s_run;
        for (int k = 0; k < wid; ++k) off += s_warp[k];
        if (keep) out[off + __popc(m & ((1u << lane) - 1u))] = v;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int k = 0; k < 8; ++k) t += s_warp[k]; s_run += t; }
        __syncthreads();
    }
}

} // namespace

bool nm_extrema_make_tma(NmBlurTma* t, const NmOctave& oc, int batch)
{
    // (x, y, level of frame): 6 * batch planes of h rows
    const unsigned long long dims[3] = {(unsigned long long)oc.w, (unsigned long long)oc.h, 6ull * batch};
    const unsigned long long strides[2] = {(unsigned long long)oc.pitch * 4, (unsigned long long)oc.level_elems * 4};
    const unsigned box[3] = {EX_P, EX_ROWS, 6};
    return nm_tma_encode_3d(t, oc.levels, dims, strides, box);
}

// extrema_kernel + refine_list_kernel over one octave; the gradient maps follow the compaction (nm_gradmap_launch).
// The window is staged by TMA only: `tma` is the descriptor nm_extrema_make_tma made for these levels.
int nm_extrema_launch(const NmOctave& oc, const NmDetectParams& dp, int batch, cudaStream_t stream, const NmBlurTma* tma)
{
    if (!tma || !tma->valid) return NM_ERR_UNSUPPORTED;
    dim3 block(32, 8), grid(nm_div_up(oc.w, EX_TW), nm_div_up(oc.h, EX_TH), batch);
    static NmDeviceOnce once;
    static std::atomic<int> ctas_cfg{2};
    if (once.first()) {
        int per_sm = 2;
        NM_CUDA_TRY(cudaFuncSetAttribute(extrema_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, EX2_SMEM));
        NM_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, extrema_kernel, 256, EX2_SMEM));
        ctas_cfg.store(per_sm < 1 ? 1 : per_sm);
        once.done();
    }
    const int n_sms = nm_sm_count(), ctas_per_sm = ctas_cfg.load();
    if (n_sms <= 0) return NM_ERR_NO_DEVICE;
    const long long n_tiles = (long long)grid.x * grid.y * grid.z;
    if (n_tiles >= (1LL << 31) / EX2_LIST || !oc.cand_n || !oc.cand) return NM_ERR_OVERFLOW;
    // 4x the resident count: co-resident CTAs do not advance evenly, and with exactly-resident persistent CTAs the
    // launch ends on half-empty SMs; the hardware hands an SM its next CTA as one retires (64 x 1080p: 1.27 -> 1.21 ms,
    // 2x 1.23, 8x 1.21; B200).
    const long long want = (long long)n_sms * ctas_per_sm * 4;
    const int ctas = (int)(n_tiles < want ? n_tiles : want);
    extrema_kernel<<<ctas, block, EX2_SMEM, stream>>>(oc, dp, tma->map, (int)grid.x, (int)grid.y, (int)n_tiles, oc.cand_n, oc.cand);
    NM_LAUNCH_CHECK();
    refine_list_kernel<<<(unsigned)nm_div_up64(n_tiles, 8), 256, 0, stream>>>(oc, dp, (int)grid.x, (int)grid.y, (int)n_tiles,
                                                                            oc.cand_n, oc.cand);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_gradmap_launch(const NmOctaveTable& tab, int batch, int dense, cudaStream_t stream)
{
    if (batch * 3 > 65535) return NM_ERR_OVERFLOW;
    for (int o = 0; o < tab.n_oct; ++o) {
        const NmOctave& oc = tab.o[o];
        const int strips_x = nm_div_up(oc.wpr, 8), nrb = nm_div_up(oc.h, NM_NEED_ROWS);
        dim3 grid(strips_x * nm_div_up(nrb, 4), batch * 3);
        gradmap_kernel<<<grid, 256, 0, stream>>>(oc, strips_x, dense);
        NM_LAUNCH_CHECK();
    }
    return NM_OK;
}

int nm_rank_launch(const NmOctaveTable& tab, int batch, int* seg_raw, cudaStream_t stream)
{
    dim3 grid(tab.n_oct * 3, batch);
    rank_kernel<<<grid, 256, 0, stream>>>(tab, seg_raw);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_plan_launch(const int* seg_raw, int* seg_cnt, int* seg_off, int* counts, int n_oct, int batch,
                   int capacity, cudaStream_t stream)
{
    plan_kernel<<<nm_div_up(batch, 64), 64, 0, stream>>>(seg_raw, seg_cnt, seg_off, counts, n_oct, batch, capacity);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_emit_launch(const NmOctave& oc, int octave_index, int n_oct, int batch,
                   const int* seg_cnt, const int* seg_off, int capacity, float4* kpts, int* meta,
                   cudaStream_t stream)
{
    dim3 grid(nm_div_up(oc.h * oc.wpr, 256), 3, batch);
    emit_kernel<<<grid, 256, 0, stream>>>(oc, octave_index, n_oct, seg_cnt, seg_off, capacity, kpts, meta);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_kprefine_launch(const NmOctaveTable& tab, const NmDetectParams& dp, int batch, int capacity, const int* counts,
                       float4* kpts, const int* meta, cudaStream_t stream)
{
    dim3 grid(nm_div_up(capacity, 256), batch);
    kprefine_kernel<<<grid, 256, 0, stream>>>(tab, dp, capacity, counts, kpts, meta);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

// ---------------------------------------------------------------------------
// C-ABI (compat granularity)
// ---------------------------------------------------------------------------
extern "C" int nm_keypoints_dense_f32(const float* dog_cur, const float* dog_down, const float* dog_up,
                                      int width, int height, float peak_threshold, float edge_threshold,
                                      float xper, float sigma_0, int num_dogs, int level, float* result4,
                                      nm_stream_t stream)
{
    if (!dog_cur || !dog_down || !dog_up || !result4 || width <= 0 || height <= 0) return NM_ERR_INVALID;
    NmDetectParams dp{peak_threshold, edge_threshold, sigma_0, num_dogs};
    dim3 block(32, 8), grid(nm_div_up(width, 32), nm_div_up(height, 8));
    keypoints_dense_linear_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
        dog_cur, dog_down, dog_up, 0, width, height, dp, xper, level, reinterpret_cast<float4*>(result4));
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_keypoints_dense_masked_f32(const float* dog_cur, const float* dog_down, const float* dog_up,
                                             unsigned long long tex_mask, int width, int height,
                                             float peak_threshold, float edge_threshold, float xper, float sigma_0,
                                             int num_dogs, int level, float* result4, nm_stream_t stream)
{
    if (!dog_cur || !dog_down || !dog_up || !result4 || width <= 0 || height <= 0) return NM_ERR_INVALID;
    NmDetectParams dp{peak_threshold, edge_threshold, sigma_0, num_dogs};
    dim3 block(32, 8), grid(nm_div_up(width, 32), nm_div_up(height, 8));
    keypoints_dense_linear_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
        dog_cur, dog_down, dog_up, (cudaTextureObject_t)tex_mask, width, height, dp, xper, level,
        reinterpret_cast<float4*>(result4));
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_keypoints_dense_tex(unsigned long long tex_cur, unsigned long long tex_mask,
                                      unsigned long long tex_down, unsigned long long tex_up, int width,
                                      int height, float peak_threshold, float edge_threshold, float xper,
                                      float sigma_0, int num_dogs, int level, float* result4,
                                      nm_stream_t stream)
{
    if (!tex_cur || !tex_down || !tex_up || !result4 || width <= 0 || height <= 0) return NM_ERR_INVALID;
    NmDetectParams dp{peak_threshold, edge_threshold, sigma_0, num_dogs};
    dim3 block(32, 8), grid(nm_div_up(width, 32), nm_div_up(height, 8));
    keypoints_dense_tex_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
        (cudaTextureObject_t)tex_cur, (cudaTextureObject_t)tex_mask, (cudaTextureObject_t)tex_down,
        (cudaTextureObject_t)tex_up, width, height, dp, xper, level, reinterpret_cast<float4*>(result4));
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_collate_f32(const float* dense4, int num_pixels, float* out4, int* count_dev,
                              nm_stream_t stream)
{
    if (!dense4 || !out4 || !count_dev || num_pixels <= 0) return NM_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    const int nblocks = nm_div_up(num_pixels, COL_CHUNK);
    int* block_counts = nullptr;
    NM_CUDA_TRY(nm_ws_alloc(&block_counts, sizeof(int) * nblocks, st));
    collate_count_kernel<<<nblocks, 256, 0, st>>>(reinterpret_cast<const float4*>(dense4), num_pixels, block_counts);
    collate_scan_kernel<<<1, 32, 0, st>>>(block_counts, nblocks, count_dev);
    collate_write_kernel<<<nblocks, 256, 0, st>>>(reinterpret_cast<const float4*>(dense4), num_pixels,
                                                  block_counts, reinterpret_cast<float4*>(out4));
    cudaError_t e = cudaGetLastError();
    cudaFreeAsync(block_counts, st);
    return nm_cuda_err(e);
}
