// nm_pyramid.cu -- Gaussian scale-space stage: separable blur, decimation, DoG
// subtraction and gradient maps.
//
// Replaces the reference's convolve<float> (gpu/kernels/convolution.cu:141-159, kernels
// :16-74 and :78-137), downsample_by_2 (gpu/kernels/downsample.cu:6-29), subtract and
// gradient (gpu/kernels/cudamath.cu:26-79).
//
// Blur design (B200): ONE kernel per level instead of the reference's row kernel +
// column kernel through a global buffer.  A CTA owns a 128x64 output tile; the
// (128+2R)x(64+2R) input window is staged in shared memory with zero fill (= the
// reference's zero padding), the row pass writes an fp32 intermediate tile to shared
// memory (the reference rounds the row result to fp32 in `buffer`, so the values are
// identical), and the column pass produces the output.  Both passes are register
// tiled (8 / 16 outputs per thread with a sliding window) so the FMA pipe, not the
// shared-memory port, is the limiter.  Each output accumulates k = -R..R in the
// reference's order with explicit fmaf, so the result is bitwise the reference's.
// Algorithmic traffic: 8 B/pixel/level (one read, one write).
// Large launches (octaves 0 and 1 of a batch) take blur_strip_kernel below, which walks down
// 128-column strips and keeps the row-pass result in a shared-memory ring, so no halo row is
// convolved twice.
//
// The input window is fetched by TMA (cp.async.bulk.tensor.3d, one elected thread, mbarrier
// completion): the hardware zero-fills everything outside the (w, h) tensor, which is
// exactly the reference's zero padding, and no thread spends issue slots or scoreboard
// stalls on the load -- two resident CTAs per SM overlap one CTA's load with the other's
// FMA phases.  Sources that TMA cannot describe (unaligned pointer or pitch) take the same
// kernel with plain loads.
#include "nm_pyramid.cuh"
#include <mutex>
#include <cstring>
#include <cstdlib>

namespace {

constexpr int kTW = 128;          // tile width  (outputs)
constexpr int kTH = 64;           // tile height (outputs)
constexpr int kThreads = 512;        // 2 CTAs per SM = 32 warps: 256-thread CTAs (16 warps) and a persistent
                                   // 512-thread CTA with double-buffered TMA windows were both ~10 % slower
constexpr int kRowPitch = kTW + 4;   // 132 == 4 (mod 32): conflict-free float4 per-row access

// TMA needs a 16-byte aligned start in the innermost dimension, so the staged window starts
// at x0 - RA with RA = R rounded up to a multiple of 4 (x0 is a multiple of 128).
__host__ __device__ constexpr int radius_aligned(int R) { return (R + 3) / 4 * 4; }
__host__ __device__ constexpr int in_pitch(int R)
{
    // >= kTW + RA + R + 3 (float4 over-read), multiple of 4, == 4 (mod 32)
    int p = kTW + radius_aligned(R) + R + 3;
    p = (p + 3) / 4 * 4;
    while (p % 32 != 4) p += 4;
    return p;
}
__host__ __device__ constexpr int blur_smem_bytes(int R)
{
    // staged window + row-pass tile + mbarrier, plus slack for the manual 128-byte alignment
    return ((kTH + 2 * R) * in_pitch(R) + (kTH + 2 * R) * kRowPitch) * (int)sizeof(float) + 16 + 128;
}

// ---- mbarrier / TMA PTX -------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LAB_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LAB_DONE_%=;\n"
        "bra LAB_WAIT_%=;\n"
        "LAB_DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int x, int y, int z)
{
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
        ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(z), "r"(smem_u32(bar))
        : "memory");
}

// d = a * (t, t) + c on both halves: one FFMA2.
__device__ __forceinline__ float2 nm_ffma2(float2 a, float t, float2 c)
{
    unsigned long long a64, b64, c64, d64;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a64) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %1};" : "=l"(b64) : "f"(t));
    asm("mov.b64 %0, {%1, %2};" : "=l"(c64) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d64) : "l"(a64), "l"(b64), "l"(c64));
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(d64));
    return d;
}

// Both passes issue their multiply-adds as FFMA2 (fma.rn.f32x2: two independent IEEE fp32 FMAs per
// instruction, a Blackwell addition): the kernel is FMA-issue bound (ncu, R = 13: FMA pipe 52 %,
// issue slots 64 % busy, DRAM at 27 %), and the paired form halves the FMA instruction count while
// every output still accumulates k = -R..R in the reference's order, so the result stays bitwise.

// ---- row pass: P outputs (P/2 pairs along x) per item, lanes walk rows (pitch == 4 mod 32) -----
template <int R, int NTHREADS>
__device__ __forceinline__ void blur_row_pass(const float* __restrict__ s_in, float* __restrict__ s_row,
                                              const float (&t)[2 * R + 1], int tid)
{
    constexpr int IH = kTH + 2 * R, SH = radius_aligned(R) - R, IP = in_pitch(R), NT = 2 * R + 1;
    constexpr int P = 8;
    constexpr int NV = (SH + P + 2 * R + 3) / 4; // float4 loads per item
    for (int it = tid; it < IH * (kTW / P); it += NTHREADS) {
        const int xs = it / IH, r = it - xs * IH;
        float wv[NV * 4 + 1];
        const float4* p4 = reinterpret_cast<const float4*>(s_in + r * IP + xs * P);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const float4 q = p4[j];
            wv[4 * j] = q.x; wv[4 * j + 1] = q.y; wv[4 * j + 2] = q.z; wv[4 * j + 3] = q.w;
        }
        wv[NV * 4] = 0.f;
        float2 acc[P / 2];
#pragma unroll
        for (int j = 0; j < P / 2; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int kk = 0; kk < NT; ++kk)
#pragma unroll
            for (int j = 0; j < P / 2; ++j)
                acc[j] = nm_ffma2(make_float2(wv[SH + 2 * j + kk], wv[SH + 2 * j + kk + 1]), t[2 * R - kk], acc[j]);
        float2* o2 = reinterpret_cast<float2*>(s_row + r * kRowPitch + xs * P);
#pragma unroll
        for (int j = 0; j < P / 2; ++j) o2[j] = acc[j];
    }
}

// ---- column pass: 2 adjacent columns x 8 rows per item, lanes walk column pairs (LDS.64) --------
template <int R, int NTHREADS>
__device__ __forceinline__ void blur_col_pass(const float* __restrict__ s_row, const NmBlurArgs& a,
                                              const float (&t)[2 * R + 1], int tid, int x0, int y0, int f)
{
    constexpr int NT = 2 * R + 1;
    constexpr int P = 8;
    float* __restrict__ dst = a.dst + (long long)f * a.dst_fstride;
    for (int it = tid; it < (kTW / 2) * (kTH / P); it += NTHREADS) {
        const int ys = it / (kTW / 2), cp = it - ys * (kTW / 2);
        const int gx = x0 + 2 * cp;
        const int gy0 = y0 + ys * P;
        if (gx >= a.w || gy0 >= a.h) continue;
        float2 wv[P + 2 * R];
        const float* p = s_row + (ys * P) * kRowPitch + 2 * cp;
#pragma unroll
        for (int j = 0; j < P + 2 * R; ++j) wv[j] = *reinterpret_cast<const float2*>(p + j * kRowPitch);
        float2 acc[P];
#pragma unroll
        for (int j = 0; j < P; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
        for (int kk = 0; kk < NT; ++kk)
#pragma unroll
            for (int j = 0; j < P; ++j) acc[j] = nm_ffma2(wv[j + kk], t[2 * R - kk], acc[j]);
        float* o = dst + (long long)gy0 * a.dst_pitch + gx;
        const bool two = gx + 1 < a.w;
        // gx is even: the pair is 8-byte aligned when the pitch is even and the image base is
        const bool vec = two && !(a.dst_pitch & 1) && !(reinterpret_cast<uintptr_t>(dst) & 7);
#pragma unroll
        for (int j = 0; j < P; ++j)
            if (gy0 + j < a.h) {
                float* oj = o + (long long)j * a.dst_pitch;
                if (vec) *reinterpret_cast<float2*>(oj) = acc[j];
                else { oj[0] = acc[j].x; if (two) oj[1] = acc[j].y; }
            }
        if (a.dst2 != nullptr && (gx >> 1) < (a.w >> 1)) {
            float* o2 = a.dst2 + (long long)f * a.dst2_fstride + (gx >> 1);
#pragma unroll
            for (int j = 0; j < P; j += 2) {
                const int hy = (gy0 + j) >> 1;       // gy0 is even (multiple of 8)
                if (hy < (a.h >> 1)) o2[(long long)hy * a.dst2_pitch] = acc[j].x;
            }
        }
    }
}

// Persistent variant for TMA-describable sources: two CTAs per SM walk the tiles of the launch.  The
// staged window is dead once the row pass has consumed it, so the TMA load of the CTA's NEXT tile is
// issued right after the row pass and lands while the column pass runs -- no second window needed.
template <int R>
__global__ void __launch_bounds__(kThreads, 2) blur_walk_kernel(const NmBlurArgs a, const __grid_constant__ CUtensorMap tmap,
                                                                int tiles_x, int tiles_y, int n_tiles)
{
    constexpr int IH = kTH + 2 * R, RA = radius_aligned(R), IP = in_pitch(R), NT = 2 * R + 1;
    extern __shared__ __align__(128) float smem[];
    float* s_in = smem;
    float* s_row = smem + IH * IP;
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_row + IH * kRowPitch);
    const int tid = threadIdx.x;
    auto tile_pos = [&](int tile, int& x0, int& y0, int& f) {
        const int tx = tile % tiles_x, r = tile / tiles_x;
        x0 = tx * kTW; y0 = (r % tiles_y) * kTH; f = r / tiles_y;
    };
    int tile = blockIdx.x;
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (tile < n_tiles) {
            int x0, y0, f;
            tile_pos(tile, x0, y0, f);
            mbar_expect_tx(bar, IH * IP * (uint32_t)sizeof(float));
            tma_load_3d(s_in, &tmap, bar, x0 - RA, y0 - R, f);
        }
    }
    float t[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) t[k] = __ldg(a.taps + k);
    __syncthreads();                           // barrier initialised before anyone polls it
    for (int k = 0; tile < n_tiles; ++k, tile += gridDim.x) {
        int x0, y0, f;
        tile_pos(tile, x0, y0, f);
        mbar_wait(bar, k & 1);
        blur_row_pass<R, kThreads>(s_in, s_row, t, tid);
        __syncthreads();                       // every thread is done with the window
        const int next = tile + gridDim.x;
        if (tid == 0 && next < n_tiles) {
            int nx0, ny0, nf;
            tile_pos(next, nx0, ny0, nf);
            mbar_expect_tx(bar, IH * IP * (uint32_t)sizeof(float));
            tma_load_3d(s_in, &tmap, bar, nx0 - RA, ny0 - R, nf);
        }
        blur_col_pass<R, kThreads>(s_row, a, t, tid, x0, y0, f);
        __syncthreads();                       // s_row is rewritten by the next row pass
    }
}

// ---- strip-walking variant: no redundant row-pass work ------------------------------------------
// blur_tile/blur_walk run the row pass over all 64 + 2R staged rows of every 64-row tile, i.e. the 2R
// halo rows are convolved twice (R = 13: 41 % more row-pass FMAs, and the FMA pipe is what bounds the
// kernel).  Here a CTA walks DOWN a 128-column strip in chunks of 64 input rows: the row pass of chunk c
// (row-pass rows i = 64c .. 64c+63, i = image row + R) goes to one half of a 128-row ring in shared
// memory, and the column pass then emits the 64 output rows whose 2R+1 inputs are now complete
// (y = 64c - 2R .. 64c + 63 - 2R), reading the 2R carried rows from the other half.  Every row-pass
// row is computed once per strip (see the work assignment at the kernel).  Arithmetic per output is
// unchanged (bitwise the reference).
constexpr int kCH = 64;            // input rows per chunk
constexpr int kRing = 128;         // ring rows (>= kCH + 2R for R <= 16; power of two)
__host__ __device__ constexpr int strip_smem_bytes(int R)
{
    return (kCH * in_pitch(R) + kRing * kRowPitch) * (int)sizeof(float) + 16 + 128;
}

template <int R>
__device__ __forceinline__ void strip_row_pass(const float* __restrict__ s_in, float* __restrict__ s_ring,
                                               const float (&t)[2 * R + 1], int tid, int ring_base, int r_begin,
                                               int y_first, int h)
{
    constexpr int SH = radius_aligned(R) - R, IP = in_pitch(R), NT = 2 * R + 1;
    constexpr int P = 8;
    constexpr int NV = (SH + P + 2 * R + 3) / 4;
    for (int it = tid; it < kCH * (kTW / P); it += kThreads) {
        const int xs = it >> 6, r = it & (kCH - 1);
        if (r < r_begin) continue;
        float2* o2 = reinterpret_cast<float2*>(s_ring + (ring_base + r) * kRowPitch + xs * P);
        const int y = y_first + r;
        if (y < 0 || y >= h) {                  // zero padding rows: the row pass of zeros
#pragma unroll
            for (int j = 0; j < P / 2; ++j) o2[j] = make_float2(0.f, 0.f);
            continue;
        }
        float wv[NV * 4 + 1];
        const float4* p4 = reinterpret_cast<const float4*>(s_in + r * IP + xs * P);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const float4 q = p4[j];
            wv[4 * j] = q.x; wv[4 * j + 1] = q.y; wv[4 * j + 2] = q.z; wv[4 * j + 3] = q.w;
        }
        wv[NV * 4] = 0.f;
        // Taps whose window offset is even read aligned register pairs (FFMA2); for the odd ones an FFMA2 would
        // need pairs that straddle two aligned pairs, which the compiler can only build with MOVs (61 per item,
        // R = 10: a quarter of the row pass's issue slots) -- those taps are issued as scalar FFMAs instead.
        float acc[P];
#pragma unroll
        for (int j = 0; j < P; ++j) acc[j] = 0.f;
#pragma unroll
        for (int kk = 0; kk < NT; ++kk) {
            if (((SH + kk) & 1) == 0) {
#pragma unroll
                for (int j = 0; j < P / 2; ++j) {
                    const float2 d = nm_ffma2(make_float2(wv[SH + 2 * j + kk], wv[SH + 2 * j + kk + 1]), t[2 * R - kk],
                                              make_float2(acc[2 * j], acc[2 * j + 1]));
                    acc[2 * j] = d.x; acc[2 * j + 1] = d.y;
                }
            } else {
#pragma unroll
                for (int j = 0; j < P; ++j) acc[j] = __fmaf_rn(wv[SH + j + kk], t[2 * R - kk], acc[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < P / 2; ++j) o2[j] = make_float2(acc[2 * j], acc[2 * j + 1]);
    }
}

template <int R, bool WRAP>
__device__ __forceinline__ void strip_col_item(const float* __restrict__ s_ring, const NmBlurArgs& a, float* __restrict__ dst,
                                               const float (&t)[2 * R + 1], int cp, int gx, int gy0, int f)
{
    constexpr int NT = 2 * R + 1;
    constexpr int P = 8;
    float2 wv[P + 2 * R];
    if (WRAP) {
        // the window crosses the end of the ring once, after n1 rows (warp-uniform)
        const int lo = gy0 & (kRing - 1), n1 = kRing - lo;
        const float* p_lo = s_ring + lo * kRowPitch + 2 * cp;
        const float* p_hi = p_lo - kRing * kRowPitch;
#pragma unroll
        for (int j = 0; j < P + 2 * R; ++j)
            wv[j] = *reinterpret_cast<const float2*>((j < n1 ? p_lo : p_hi) + j * kRowPitch);
    } else {
        const float* p = s_ring + (gy0 & (kRing - 1)) * kRowPitch + 2 * cp;
#pragma unroll
        for (int j = 0; j < P + 2 * R; ++j) wv[j] = *reinterpret_cast<const float2*>(p + j * kRowPitch);
    }
    float2 acc[P];
#pragma unroll
    for (int j = 0; j < P; ++j) acc[j] = make_float2(0.f, 0.f);
#pragma unroll
    for (int kk = 0; kk < NT; ++kk)
#pragma unroll
        for (int j = 0; j < P; ++j) acc[j] = nm_ffma2(wv[j + kk], t[2 * R - kk], acc[j]);
    float* o = dst + (long long)gy0 * a.dst_pitch + gx;
    const bool two = gx + 1 < a.w;
    const bool vec = two && !(a.dst_pitch & 1) && !(reinterpret_cast<uintptr_t>(dst) & 7);
#pragma unroll
    for (int j = 0; j < P; ++j)
        if (gy0 + j >= 0 && gy0 + j < a.h) {
            float* oj = o + (long long)j * a.dst_pitch;
            if (vec) *reinterpret_cast<float2*>(oj) = acc[j];
            else { oj[0] = acc[j].x; if (two) oj[1] = acc[j].y; }
        }
    if (a.dst2 != nullptr && (gx >> 1) < (a.w >> 1)) {
        float* o2 = a.dst2 + (long long)f * a.dst2_fstride + (gx >> 1);
#pragma unroll
        for (int j = 0; j < P; j += 2) {
            const int gy = gy0 + j;              // gy0 is even (64c - 2R + 8 ys)
            if (gy >= 0 && (gy >> 1) < (a.h >> 1)) o2[(long long)(gy >> 1) * a.dst2_pitch] = acc[j].x;
        }
    }
}

// Work assignment (strips = tiles_x * batch, `chunks` per strip, G = gridDim.x persistent CTAs): in round r <
// full_rounds CTA b walks the WHOLE strip r*G + b, so the strips in flight at any time are neighbours in the
// image and the RA + R halo columns a strip shares with its neighbours are L2 hits (a flat split of the chunk
// list had every CTA ~3 strips away from the next one: 12 % more DRAM traffic than the algorithmic bytes); the
// strips left over after the full rounds are split evenly as one flat chunk list, CTA b taking the b-th piece,
// which may start inside a strip (then it is preceded by the row pass of the previous chunk's last 2R rows).
template <int R>
__global__ void __launch_bounds__(kThreads, 2) blur_strip_kernel(const NmBlurArgs a, const __grid_constant__ CUtensorMap tmap,
                                                                 int tiles_x, int chunks, int full_rounds, long long total)
{
    constexpr int RA = radius_aligned(R), IP = in_pitch(R), NT = 2 * R + 1;
    extern __shared__ __align__(128) float smem[];
    float* s_in = smem;                        // [kCH][IP]
    float* s_ring = smem + kCH * IP;           // [kRing][kRowPitch]
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_ring + kRing * kRowPitch);
    const int tid = threadIdx.x;
    const long long G = gridDim.x, rem0 = (long long)full_rounds * G * chunks, rem = total - rem0;
    // piece ri of this CTA: chunks [g0, g1) of the strip-major chunk list
    auto piece = [&](int ri, long long& g0, long long& g1) {
        if (ri < full_rounds) { g0 = ((long long)ri * G + blockIdx.x) * chunks; g1 = g0 + chunks; }
        else { g0 = rem0 + rem * blockIdx.x / G; g1 = rem0 + rem * (blockIdx.x + 1) / G; }
    };
    auto locate = [&](long long g, int& c, int& tx, int& f) {
        const int s = (int)(g / chunks);
        c = (int)(g - (long long)s * chunks); tx = s % tiles_x; f = s / tiles_x;
    };
    auto issue = [&](int cc, int txx, int ff) {
        mbar_expect_tx(bar, kCH * IP * (uint32_t)sizeof(float));
        tma_load_3d(s_in, &tmap, bar, txx * kTW - RA, cc * kCH - R, ff);
    };
    int ri = 0;
    long long g0, g1;
    piece(ri, g0, g1);
    if (g0 >= g1) {
        if (ri >= full_rounds) return;         // (only the remainder piece can be empty)
    }
    long long g = (g0 % chunks) ? g0 - 1 : g0;
    int c, tx, f;
    locate(g, c, tx, f);
    if (tid == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        issue(c, tx, f);
    }
    float t[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) t[k] = __ldg(a.taps + k);
    __syncthreads();
    for (uint32_t phase = 0;; phase ^= 1) {
        const bool pre = g < g0;
        // the chunk after this one: down the strip inside a piece, else the first chunk of the next piece
        long long ng = g + 1, ng0 = g0, ng1 = g1;
        int nri = ri, nc = c + 1, ntx = tx, nf = f;
        bool more = true;
        if (ng < g1) {
            if (nc == chunks) { nc = 0; if (++ntx == tiles_x) { ntx = 0; ++nf; } }
        } else if (ri < full_rounds) {
            nri = ri + 1;
            piece(nri, ng0, ng1);
            more = ng0 < ng1;
            if (more) {
                ng = (ng0 % chunks) ? ng0 - 1 : ng0;
                locate(ng, nc, ntx, nf);
            }
        } else more = false;
        mbar_wait(bar, phase);
        if (a.src_bgra) {
            // the staged words are BGRA pixels: grey values in place (zero fill outside the frame stays 0)
            float4* w4 = reinterpret_cast<float4*>(s_in);
            for (int i = tid; i < kCH * IP / 4; i += kThreads) {
                const float4 q = w4[i];
                w4[i] = make_float4(nm_gray_from_bgra(__float_as_uint(q.x)), nm_gray_from_bgra(__float_as_uint(q.y)),
                                    nm_gray_from_bgra(__float_as_uint(q.z)), nm_gray_from_bgra(__float_as_uint(q.w)));
            }
            // these generic-proxy writes are followed by the next chunk's TMA write to the same bytes (async proxy)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
        }
        strip_row_pass<R>(s_in, s_ring, t, tid, (c & 1) * kCH, pre ? kCH - 2 * R : 0, c * kCH - R, a.h);
        __syncthreads();                       // window consumed, ring rows visible
        if (tid == 0 && more) issue(nc, ntx, nf);
        if (!pre) {
            float* __restrict__ dst = a.dst + (long long)f * a.dst_fstride;
            for (int it = tid; it < (kTW / 2) * (kCH / 8); it += kThreads) {
                const int ys = it / (kTW / 2), cp = it - ys * (kTW / 2);
                const int gx = tx * kTW + 2 * cp;
                const int gy0 = c * kCH - 2 * R + ys * 8;
                if (gx >= a.w || gy0 + 8 <= 0 || gy0 >= a.h) continue;
                if ((gy0 & (kRing - 1)) + 8 + 2 * R <= kRing) strip_col_item<R, false>(s_ring, a, dst, t, cp, gx, gy0, f);
                else strip_col_item<R, true>(s_ring, a, dst, t, cp, gx, gy0, f);
            }
        }
        if (!more) break;
        g = ng; g0 = ng0; g1 = ng1; ri = nri; c = nc; tx = ntx; f = nf;
        __syncthreads();                       // the next row pass overwrites ring rows this pass read
    }
}

// ---- streaming variant: warp-specialised, no CTA-wide barrier in the steady state ---------------
// blur_strip_kernel's CTAs alternate a row-pass phase and a column-pass phase between __syncthreads(): every phase
// opens with a burst of shared-memory loads and closes with a burst of stores, and all warps of a CTA reach them
// together, so the FMA pipe -- the unit that bounds the blur -- idles 40-50 % of the time (ncu, round 2).  Here a CTA
// of four warps walks down a 128-column strip in GROUPS of kGR rows with the two passes running concurrently:
//   producers (2 warps)  row pass of group n from TMA stage n % kNS into ring slot n % kNG; lane 0 of the first one
//                        also issues the TMA loads, kNS - 1 groups ahead
//   consumers (2 warps)  column pass in SCATTER form: a lane owns one column pair and walks down the rows holding
//                        the 2R+1 outputs in flight in registers -- input row i adds in[i] * t[2R-kk] to output
//                        i - kk for kk = 0..2R, so every output still accumulates its taps in the reference's order
//                        (bitwise the reference), each row-pass value is read from shared memory exactly once
//                        (one LDS.64 per 2R+1 FFMA2), and one output row completes per input row
// with mbarrier full/empty pairs per stage and per ring slot as the only synchronisation.  Work split, halo reuse
// through L2 and the piece rule are blur_strip_kernel's, in units of groups; a piece that starts inside a strip is
// preceded by ceil(2R / kGR) groups whose outputs are not stored (they fill the accumulators).
// Measured (64 x 1080p, B200; pyramid stage of the step, blur_strip_kernel = 2.25 ms):
//   8-row groups, 3 + 3 buffers, roles rotating over the SM sub-partitions   2.29 ms
//   the same, fixed roles (warps 0-1 produce, 2-3 consume in every CTA)       2.18 ms   (each sub-partition's
//                                                                             instruction cache sees one role)
//   16-row groups, 2 + 2 buffers                                              2.06 ms   (half the hand-overs)
//   deeper rings (3 or 4 slots) or 3 stages: no change / slower (fewer resident CTAs)
//   oversubscribed launch, two CTAs per strip (see launch_tile)               1.96 ms
// Per launch (octave 0, ncu, final): R = 5 188 us, 7 201, 8 (+ decimated copy) 248, 10 247, 13 312 against
// 216 / 245 / 282 / 303 / 368 for blur_strip_kernel; the HBM floor of a level is 165 us, the FMA floor of R = 13 192 us.
constexpr int kGR = 16;            // rows per group
constexpr int kNS = 2;             // TMA stages
constexpr int kNG = 2;             // ring slots (2 + 2 of 16 rows: 38 KB of shared memory per CTA, 5 CTAs per SM)
constexpr int kStreamThreads = 128;
constexpr int kStreamPieces = 32;  // pieces per CTA the schedule table holds
constexpr int kStreamMaxR = 13;    // 2R+1 float2 accumulators + the row-pass window fit 128 registers up to here
__host__ __device__ constexpr int stream_smem_bytes(int R)
{
    return (kNS * kGR * in_pitch(R) + kNG * kGR * kRowPitch) * (int)sizeof(float) + 2 * (kNS + kNG) * 8 +
           kStreamPieces * 32 + 128;
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

struct StreamPiece { int gs, g0, g1, c, tx, f, pad0, pad1; };
struct StreamTaps { float v[33]; };      // by value: kernel parameters live in the constant bank, which the warp-
                                          // specialised code can name as an FFMA operand (taps loaded from global memory
                                          // ended up in 2R+1 ordinary registers there and spilled for R >= 11)   // groups [gs, g1) are walked, [g0, g1) are owned

struct StreamWalk {
    int g, g0, g1, ri, c, tx, f;
    bool valid;
    __device__ __forceinline__ void enter(const StreamPiece* tab, int n_pieces)
    {
        valid = ri < n_pieces;
        if (!valid) return;
        const int4 a = *reinterpret_cast<const int4*>(&tab[ri].gs);
        const int2 b = *reinterpret_cast<const int2*>(&tab[ri].tx);
        g = a.x; g0 = a.y; g1 = a.z; c = a.w; tx = b.x; f = b.y;
    }
    __device__ __forceinline__ void next(const StreamPiece* tab, int n_pieces, int cg, int tiles_x)
    {
        if (++g < g1) {
            if (++c == cg) { c = 0; if (++tx == tiles_x) { tx = 0; ++f; } }
        } else { ++ri; enter(tab, n_pieces); }
    }
};

// one row-pass item: 8 outputs of one row (the arithmetic of strip_row_pass)
template <int R>
__device__ __forceinline__ void stream_row_item(const float* __restrict__ in, float* __restrict__ out,
                                                const float* __restrict__ t)
{
    constexpr int SH = radius_aligned(R) - R, NT = 2 * R + 1;
    constexpr int P = 8;
    constexpr int NV = (SH + P + 2 * R + 3) / 4;
    float wv[NV * 4 + 1];
    const float4* p4 = reinterpret_cast<const float4*>(in);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const float4 q = p4[j];
        wv[4 * j] = q.x; wv[4 * j + 1] = q.y; wv[4 * j + 2] = q.z; wv[4 * j + 3] = q.w;
    }
    wv[NV * 4] = 0.f;
    float acc[P];
#pragma unroll
    for (int j = 0; j < P; ++j) acc[j] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NT; ++kk) {
        if (((SH + kk) & 1) == 0) {
#pragma unroll
            for (int j = 0; j < P / 2; ++j) {
                const float2 d = nm_ffma2(make_float2(wv[SH + 2 * j + kk], wv[SH + 2 * j + kk + 1]), t[2 * R - kk],
                                          make_float2(acc[2 * j], acc[2 * j + 1]));
                acc[2 * j] = d.x; acc[2 * j + 1] = d.y;
            }
        } else {
#pragma unroll
            for (int j = 0; j < P; ++j) acc[j] = __fmaf_rn(wv[SH + j + kk], t[2 * R - kk], acc[j]);
        }
    }
    float4* o4 = reinterpret_cast<float4*>(out);
    o4[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    o4[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
}

__host__ __device__ constexpr int stream_min_ctas(int R) { return R <= 10 ? 5 : 4; }

template <int R, bool DST2>
__global__ void __launch_bounds__(kStreamThreads, stream_min_ctas(R)) blur_stream_kernel(const NmBlurArgs a, const __grid_constant__ CUtensorMap tmap,
                                                                         const __grid_constant__ StreamTaps taps,
                                                                         int tiles_x, int cg, int full_rounds, int total)
{
    constexpr int RA = radius_aligned(R), IP = in_pitch(R), NT = 2 * R + 1;
    constexpr int PRE = (2 * R + kGR - 1) / kGR;
    extern __shared__ __align__(128) float smem[];
    float* s_in = smem;                                  // [kNS][kGR][IP]
    float* s_ring = smem + kNS * kGR * IP;               // [kNG][kGR][kRowPitch]
    uint64_t* in_full = reinterpret_cast<uint64_t*>(s_ring + kNG * kGR * kRowPitch);
    uint64_t* in_empty = in_full + kNS;
    uint64_t* ring_full = in_empty + kNS;
    uint64_t* ring_empty = ring_full + kNG;
    StreamPiece* tab = reinterpret_cast<StreamPiece*>(ring_empty + kNG);
    __shared__ int s_steps;
    __shared__ float s_taps[NT];
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < NT) s_taps[tid] = taps.v[tid];
    // full_rounds < 0: oversubscribed launch, -full_rounds CTAs per strip, CTA b = part b / strips of strip b % strips
    const int n_pieces = full_rounds < 0 ? 1 : full_rounds + 1;   // <= kStreamPieces (launcher); the last one may be empty
    if (tid < n_pieces) {
        const long long G = gridDim.x, rem0 = (long long)full_rounds * G * cg, rem = total - rem0;
        long long g0, g1;
        if (full_rounds < 0) {
            const int parts = -full_rounds, strips = total / cg, sx = blockIdx.x % strips, px = blockIdx.x / strips;
            g0 = (long long)sx * cg + (long long)px * cg / parts; g1 = (long long)sx * cg + (long long)(px + 1) * cg / parts;
        } else if (tid < full_rounds) { g0 = ((long long)tid * G + blockIdx.x) * cg; g1 = g0 + cg; }
        else { g0 = rem0 + rem * blockIdx.x / G; g1 = rem0 + rem * (blockIdx.x + 1) / G; }
        const int s = (int)(g0 / cg), c0 = (int)(g0 - (long long)s * cg), pre = min(PRE, c0);
        StreamPiece p;
        p.gs = (int)g0 - pre; p.g0 = (int)g0; p.g1 = (int)g1; p.c = c0 - pre; p.tx = s % tiles_x; p.f = s / tiles_x;
        p.pad0 = p.pad1 = 0;
        if (g0 >= g1) p.gs = p.g0 = p.g1 = 0;            // empty remainder piece: no steps
        tab[tid] = p;
    }
    if (tid == 0) {
        for (int i = 0; i < kNS; ++i) { mbar_init(in_full + i, 1); mbar_init(in_empty + i, 2); }
        for (int i = 0; i < kNG; ++i) { mbar_init(ring_full + i, 2); mbar_init(ring_empty + i, 2); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        int n = 0;
        for (int i = 0; i < n_pieces; ++i) n += tab[i].g1 - tab[i].gs;
        s_steps = n;
    }
    __syncthreads();
    const int n_steps = s_steps;
    if (n_steps == 0) return;
    // an empty remainder piece is always the last one: walking stops there
    const int live_pieces = (tab[n_pieces - 1].g1 > tab[n_pieces - 1].gs) ? n_pieces : n_pieces - 1;

    const float* __restrict__ t = taps.v;

    // fixed roles: warps 0-1 produce, 2-3 consume in every CTA (each SM sub-partition's instruction cache sees one role)
    const int role = (tid >> 5) & 3;
    if (role < 2) {
        // ---------------- producer: row pass ----------------
        StreamWalk wi;                                    // TMA cursor (meaningful in role 0 only)
        wi.ri = 0; wi.enter(tab, live_pieces);
        int issued = 0;
        auto issue = [&]() {
            const int slot = issued % kNS, use = issued / kNS;
            if (lane == 0) {
                if (use >= 1) mbar_wait(in_empty + slot, (use - 1) & 1);
                mbar_expect_tx(in_full + slot, kGR * IP * (uint32_t)sizeof(float));
                tma_load_3d(s_in + slot * kGR * IP, &tmap, in_full + slot, wi.tx * kTW - RA, wi.c * kGR - R, wi.f);
            }
            wi.next(tab, live_pieces, cg, tiles_x);
            ++issued;
        };
        if (role == 0)
            for (int i = 0; i < kNS - 1 && issued < n_steps; ++i) issue();
        const int r = lane & (kGR - 1), xs0 = lane / kGR + (32 / kGR) * role;   // items: rows r, segments xs0 + (64 / kGR) k
        for (int n = 0; n < n_steps; ++n) {
            if (role == 0) {
                if (issued < n_steps) issue();
                __syncwarp();
            }
            const int slot = n % kNS, q = n % kNG;
            mbar_wait(in_full + slot, (n / kNS) & 1);
            if (n >= kNG) mbar_wait(ring_empty + q, ((n / kNG) - 1) & 1);
            const float* in = s_in + (slot * kGR + r) * IP + xs0 * 8;
            float* out = s_ring + (q * kGR + r) * kRowPitch + xs0 * 8;
#pragma unroll 1
            for (int k = 0; k < kGR / 4; ++k) stream_row_item<R>(in + (512 / kGR) * k, out + (512 / kGR) * k, t);
            __syncwarp();
            if (lane == 0) { mbar_arrive(in_empty + slot); mbar_arrive(ring_full + q); }
        }
    } else {
        // ---------------- consumer: column pass, scatter form ----------------
        // The 2R+1 accumulators rotate through the roles "starts with this row" ... "completes with this row", so the
        // row step is unrolled 2R+1 times with static register names (NM_STREAM_STEP(U): the step in which acc[U]
        // starts).  A group is 16 rows and 2R+1 is odd, so a group begins at any phase: the group loop re-enters the
        // unrolled sequence through a switch (Duff's device).  The group hand-over is outside the sequence, which
        // keeps the hot code contiguous and at (2R+1) x ~38 instructions within the 32 KB instruction cache -- inlined
        // into every step it was 53 KB for R = 13 and 18 % of the warp samples were instruction-fetch stalls.
        const int cp = (role - 2) * 32 + lane;
        StreamWalk wk;
        wk.ri = 0; wk.enter(tab, live_pieces);
        float2 acc[NT];
#pragma unroll
        for (int j = 0; j < NT; ++j) acc[j] = make_float2(0.f, 0.f);
        // taps in ordinary registers, read from shared memory so that the compiler cannot re-materialise them: as
        // parameters it re-read them into uniform registers in every step of the switch (8 LDCU per 27 FFMA2)
        float tr[NT];
#pragma unroll
        for (int k = 0; k < NT; ++k) tr[k] = s_taps[k];
        int phase = 0;
        for (int n = 0; n < n_steps; ++n) {
            const int q = n % kNG;
            mbar_wait(ring_full + q, (n / kNG) & 1);
            const float* rp = s_ring + (q * kGR) * kRowPitch + 2 * cp;   // current input row, this lane's column pair
            const int gx = wk.tx * kTW + 2 * cp;                         // even, and so is a.w (launcher): gx + 1 < a.w too
            const int ylim = (wk.g >= wk.g0 && gx < a.w) ? a.h : 0;      // this lane stores rows 0 <= y < ylim
            int y = wk.c * kGR - 2 * R;                                  // the output row that completes with the current input row
            float* orow = a.dst + (long long)wk.f * a.dst_fstride + (long long)y * a.dst_pitch + gx;
            const int half_pitch2 = a.dst2_pitch >> 1;                   // dst2_pitch is even (launcher)
            float* o2half = DST2 ? a.dst2 + (long long)wk.f * a.dst2_fstride + (long long)y * half_pitch2 + (gx >> 1)
                                 : nullptr;                              // &dst2[f][y / 2][gx / 2] when y is even
            float2 v = *reinterpret_cast<const float2*>(rp);
            int left = kGR;
#define NM_STREAM_STEP(U)                                                                                              \
            case U:                                                                                                    \
                if constexpr (U < NT) {                                                                                \
                    /* the row after the group's last one is read too (inside the buffer) and never used */          \
                    const float2 vn = *reinterpret_cast<const float2*>(rp + kRowPitch);                                \
                    acc[U] = nm_ffma2(v, tr[2 * R], make_float2(0.f, 0.f));                                            \
                    _Pragma("unroll") for (int kk = 1; kk < NT; ++kk)                                                  \
                        acc[(U - kk + NT) % NT] = nm_ffma2(v, tr[2 * R - kk], acc[(U - kk + NT) % NT]);                \
                    if ((unsigned)y < (unsigned)ylim) *reinterpret_cast<float2*>(orow) = acc[(U + 1) % NT];            \
                    if (DST2) {              /* o2half advances half a decimated row per row: right on even y */     \
                        if (!(y & 1) && (unsigned)y < (unsigned)(ylim & ~1)) *o2half = acc[(U + 1) % NT].x;            \
                        o2half += half_pitch2;                                                                         \
                    }                                                                                                  \
                    ++y; orow += a.dst_pitch; rp += kRowPitch; v = vn;                                                 \
                    if (--left == 0) { phase = (U + 1) % NT; break; }                                                  \
                }
            switch (phase) {
                for (;;) {
                    NM_STREAM_STEP(0) NM_STREAM_STEP(1) NM_STREAM_STEP(2) NM_STREAM_STEP(3) NM_STREAM_STEP(4)
                    NM_STREAM_STEP(5) NM_STREAM_STEP(6) NM_STREAM_STEP(7) NM_STREAM_STEP(8) NM_STREAM_STEP(9)
                    NM_STREAM_STEP(10) NM_STREAM_STEP(11) NM_STREAM_STEP(12) NM_STREAM_STEP(13) NM_STREAM_STEP(14)
                    NM_STREAM_STEP(15) NM_STREAM_STEP(16) NM_STREAM_STEP(17) NM_STREAM_STEP(18) NM_STREAM_STEP(19)
                    NM_STREAM_STEP(20) NM_STREAM_STEP(21) NM_STREAM_STEP(22) NM_STREAM_STEP(23) NM_STREAM_STEP(24)
                    NM_STREAM_STEP(25) NM_STREAM_STEP(26)
                }
            }
#undef NM_STREAM_STEP
            __syncwarp();
            if (lane == 0) mbar_arrive(ring_empty + q);
            wk.next(tab, live_pieces, cg, tiles_x);
        }
    }
}

template <int R, bool TMA>
__global__ void __launch_bounds__(kThreads, 2) blur_tile_kernel(const NmBlurArgs a, const __grid_constant__ CUtensorMap tmap)
{
    constexpr int IH = kTH + 2 * R;          // rows staged
    constexpr int RA = radius_aligned(R);    // staged column 0 is image column x0 - RA
    constexpr int SH = RA - R;               // first column a row-pass window really needs
    constexpr int IW = kTW + RA + R;         // columns staged
    constexpr int IP = in_pitch(R);
    constexpr int NT = 2 * R + 1;
    // the kernel has no static shared memory, so the dynamic window starts at the 128-byte aligned
    // base the attribute asks for (TMA destination alignment); no pointer arithmetic on the base,
    // which would turn every LDS/STS below into a generic LD/ST
    extern __shared__ __align__(128) float smem[];
    float* s_in = smem;
    float* s_row = smem + IH * IP;
    uint64_t* bar = reinterpret_cast<uint64_t*>(s_row + IH * kRowPitch);

    const int tid = threadIdx.x;
    const int x0 = blockIdx.x * kTW, y0 = blockIdx.y * kTH, f = blockIdx.z;

    if (TMA) {
        // ---- stage the input window by TMA; out-of-tensor elements arrive as +0 -------
        if (tid == 0) {
            mbar_init(bar, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
            mbar_expect_tx(bar, IH * IP * (uint32_t)sizeof(float));
            tma_load_3d(s_in, &tmap, bar, x0 - RA, y0 - R, f);
        }
    }
    float t[NT];
#pragma unroll
    for (int k = 0; k < NT; ++k) t[k] = __ldg(a.taps + k);
    if (TMA) {
        __syncthreads();                       // barrier initialised before anyone polls it
        mbar_wait(bar, 0);
    } else {
        // ---- plain loads, zero fill outside the image ---------------------------------
        const float* __restrict__ src = a.src + (long long)f * a.src_fstride;
        for (int i = tid; i < IH * IP; i += kThreads) {
            const int r = i / IP, c = i - r * IP;
            const int gy = y0 - R + r, gx = x0 - RA + c;
            float v = 0.f;
            if (c < IW && gy >= 0 && gy < a.h && gx >= 0 && gx < a.w)
                v = __ldg(src + (long long)gy * a.src_pitch + gx);
            s_in[i] = v;
        }
        __syncthreads();
    }

    blur_row_pass<R, kThreads>(s_in, s_row, t, tid);
    __syncthreads();
    blur_col_pass<R, kThreads>(s_row, a, t, tid, x0, y0, f);
}

// Generic radius (R > 16): two plain kernels through `scratch`, same arithmetic.
__global__ void blur_rows_generic(const NmBlurArgs a)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    if (x >= a.w) return;
    const float* row = a.src + (long long)f * a.src_fstride + (long long)y * a.src_pitch;
    const int R = a.radius;
    float sum = 0.f;
    for (int k = -R; k <= R; ++k) {
        const int xx = x + k;
        const float d = (xx >= 0 && xx < a.w) ? __ldg(row + xx) : 0.f;
        sum = __fmaf_rn(d, __ldg(a.taps + (R - k)), sum);
    }
    a.scratch[((long long)f * a.h + y) * a.w + x] = sum;
}
__global__ void blur_cols_generic(const NmBlurArgs a)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, f = blockIdx.z;
    if (x >= a.w) return;
    const float* img = a.scratch + (long long)f * a.h * a.w;
    const int R = a.radius;
    float sum = 0.f;
    for (int k = -R; k <= R; ++k) {
        const int yy = y + k;
        const float d = (yy >= 0 && yy < a.h) ? img[(long long)yy * a.w + x] : 0.f;
        sum = __fmaf_rn(d, __ldg(a.taps + (R - k)), sum);
    }
    a.dst[(long long)f * a.dst_fstride + (long long)y * a.dst_pitch + x] = sum;
    if (a.dst2 != nullptr && !(x & 1) && !(y & 1) && (x >> 1) < (a.w >> 1) && (y >> 1) < (a.h >> 1))
        a.dst2[(long long)f * a.dst2_fstride + (long long)(y >> 1) * a.dst2_pitch + (x >> 1)] = sum;
}

int sm_count() { return nm_sm_count(); }

// The strip-walking kernel is taken for TMA-describable sources with enough chunks: below ~8 chunks per CTA the
// lead-in row pass of a piece that starts inside a strip costs more than the tile kernels' halo rows.
// NM_BLUR_STRIP_MIN overrides the threshold (test hook: the tests force 1).
bool strip_eligible(const NmBlurArgs& a, const NmBlurTma* tma)
{
    const int n_sms = sm_count();
    if (!tma || !tma->valid || !tma->valid_strip || n_sms <= 0 || a.radius < 1 || a.radius > 16) return false;
    static const long long strip_min_env = getenv("NM_BLUR_STRIP_MIN") ? atoll(getenv("NM_BLUR_STRIP_MIN")) : -1;
    const long long strip_min = strip_min_env >= 0 ? strip_min_env : 16LL * n_sms;
    const long long strips = (long long)nm_div_up(a.w, kTW) * a.batch;
    const long long total = strips * nm_div_up(a.h + 2 * a.radius, kCH);
    return total >= strip_min && strips < (1LL << 31);
}

// The streaming kernel takes what the strip kernel takes when the destination allows 8-byte stores, the source is
// float (BGRA conversion stays with the strip kernel) and the CTA's piece table fits.  NM_BLUR_STREAM=0 disables it
// (test hook: the tests use it to reach the strip kernel).
bool stream_eligible(const NmBlurArgs& a, const NmBlurTma* tma)
{
    static const bool off = getenv("NM_BLUR_STREAM") != nullptr && atoi(getenv("NM_BLUR_STREAM")) == 0;
    if (off || !strip_eligible(a, tma) || !tma->valid_stream || a.src_bgra || a.taps_host == nullptr) return false;
    if (a.radius > kStreamMaxR || (a.w & 1)) return false;
    if ((a.dst_pitch & 1) || (a.dst_fstride & 1) || (reinterpret_cast<uintptr_t>(a.dst) & 7)) return false;
    if (a.dst2 != nullptr && (a.dst2_pitch & 1)) return false;
    const long long strips = (long long)nm_div_up(a.w, kTW) * a.batch, G = (long long)stream_min_ctas(a.radius) * sm_count();
    const long long total = strips * nm_div_up(a.h + 2 * a.radius, kGR);
    return total < (1LL << 31) && strips / G + 1 <= kStreamPieces;
}

template <int R>
int launch_tile(const NmBlurArgs& a, cudaStream_t stream, const NmBlurTma* tma)
{
    if (a.src_bgra && !strip_eligible(a, tma)) return NM_ERR_INVALID;     // only the strip kernel converts
    static NmDeviceOnce once;
    constexpr int smem = blur_smem_bytes(R);
    if (once.first()) {
        NM_CUDA_TRY(cudaFuncSetAttribute(blur_tile_kernel<R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        NM_CUDA_TRY(cudaFuncSetAttribute(blur_tile_kernel<R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        NM_CUDA_TRY(cudaFuncSetAttribute(blur_walk_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        NM_CUDA_TRY(cudaFuncSetAttribute(blur_strip_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, strip_smem_bytes(R)));
        once.done();
    }
    dim3 grid(nm_div_up(a.w, kTW), nm_div_up(a.h, kTH), a.batch);
    if (tma && tma->valid) {
        const int n_sms = nm_sm_count();
        if (n_sms <= 0) return NM_ERR_NO_DEVICE;
        const long long n_tiles = (long long)grid.x * grid.y * grid.z;
        const int chunks = nm_div_up(a.h + 2 * R, kCH);
        const long long total = (long long)grid.x * a.batch * chunks;
        if constexpr (R <= kStreamMaxR) if (stream_eligible(a, tma)) {
            static NmDeviceOnce once_stream;
            if (once_stream.first()) {
                NM_CUDA_TRY(cudaFuncSetAttribute(blur_stream_kernel<R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 stream_smem_bytes(R)));
                NM_CUDA_TRY(cudaFuncSetAttribute(blur_stream_kernel<R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                                 stream_smem_bytes(R)));
                once_stream.done();
            }
            const long long n_strips = (long long)grid.x * a.batch;
            // Co-resident CTAs do not advance evenly (the same work takes 45 to 105 us), so a launch
            // of exactly-resident persistent CTAs ends with a long tail of half-empty SMs.  When there are enough strips
            // the launch is OVERSUBSCRIBED instead: P CTAs per strip (part b / strips of strip b % strips, so CTAs that
            // start together are neighbours in the image), about 2.5x the resident count, and the hardware hands an SM
            // its next CTA as soon as one retires.  64 x 1080p (B200): P = 2, pyramid 2.06 -> 1.96 ms (P = 1: 2.11, 3: 2.00).
            const int cg = nm_div_up(a.h + 2 * R, kGR);
            const long long resident = (long long)stream_min_ctas(R) * n_sms;
            // smallest P that reaches 2.5x the resident count with parts of >= 16 groups (the lead-in of a part is
            // ceil(2R / 16) groups), else the largest such P that still reaches 1.5x, else the persistent split
            int parts = 0;
            for (int p = 1; p <= 8 && cg >= 16 * p; ++p) {
                if (2 * n_strips * p >= 3 * resident) parts = p;
                if (2 * n_strips * p >= 5 * resident) break;
            }
            const bool over = parts > 0 && n_strips * parts > resident && n_strips * parts < (1 << 20) && cg >= 4 * parts;
            const int G = over ? (int)(n_strips * parts) : (int)resident;
            const int rounds_arg = over ? -parts : (int)(n_strips / G);
            StreamTaps tp;
            memset(&tp, 0, sizeof(tp));
            memcpy(tp.v, a.taps_host, sizeof(float) * (2 * R + 1));
            if (a.dst2 != nullptr)
                blur_stream_kernel<R, true><<<G, kStreamThreads, stream_smem_bytes(R), stream>>>(
                        a, tma->map_stream, tp, (int)grid.x, cg, rounds_arg, (int)(n_strips * cg));
            else
                blur_stream_kernel<R, false><<<G, kStreamThreads, stream_smem_bytes(R), stream>>>(
                    a, tma->map_stream, tp, (int)grid.x, cg, rounds_arg, (int)(n_strips * cg));
            NM_LAUNCH_CHECK();
            return NM_OK;
        }
        if (strip_eligible(a, tma)) {
            const long long n_strips = (long long)grid.x * a.batch;
            blur_strip_kernel<R><<<2 * n_sms, kThreads, strip_smem_bytes(R), stream>>>(a, tma->map_strip, (int)grid.x, chunks,
                                                                                      (int)(n_strips / (2 * n_sms)), total);
        } else if (n_tiles >= 4LL * n_sms && n_tiles < (1LL << 31))
            blur_walk_kernel<R><<<2 * n_sms, kThreads, smem, stream>>>(a, tma->map, (int)grid.x, (int)grid.y, (int)n_tiles);
        else
            blur_tile_kernel<R, true><<<grid, kThreads, smem, stream>>>(a, tma->map);
    } else {
        CUtensorMap dummy;
        memset(&dummy, 0, sizeof(dummy));
        blur_tile_kernel<R, false><<<grid, kThreads, smem, stream>>>(a, dummy);
    }
    NM_LAUNCH_CHECK();
    return NM_OK;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encoder()
{
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            cudaGetLastError();
    });
    return fn;
}

__global__ void downsample2_kernel(float* __restrict__ dst, int dw, int dh, int dpitch,
                                   long long dfstride, const float* __restrict__ src, int spitch,
                                   long long sfstride)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    const int f = blockIdx.z;
    if (x >= dw || y >= dh) return;
    dst[f * dfstride + (long long)y * dpitch + x] =
        __ldg(src + f * sfstride + (long long)(2 * y) * spitch + 2 * x);
}

__global__ void subtract_kernel(const float* __restrict__ A, const float* __restrict__ B,
                                float* __restrict__ C, long long n)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) C[i] = __fsub_rn(__ldg(A + i), __ldg(B + i));
}

__global__ void gradient_kernel(const float* __restrict__ src, float2* __restrict__ grad, int w, int h)
{
    const int x = blockIdx.x * blockDim.x + threadIdx.x;
    const int y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x < 1 || x >= w - 1 || y < 1 || y >= h - 1) return;
    const long long i = (long long)y * w + x;
    grad[i] = nm_gradient_at(__ldg(src + i + 1), __ldg(src + i - 1), __ldg(src + i + w), __ldg(src + i - w));
}

} // namespace

bool nm_tma_encode_3d(NmBlurTma* t, const float* base, const unsigned long long dims[3],
                      const unsigned long long strides_bytes[2], const unsigned box[3])
{
    t->valid = t->valid_strip = t->valid_stream = false;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (strides_bytes[0] & 15) || (strides_bytes[1] & 15)) return false;
    EncodeTiledFn enc = get_encoder();
    if (!enc) return false;
    const cuuint64_t d[3] = {dims[0], dims[1], dims[2]};
    const cuuint64_t st[2] = {strides_bytes[0], strides_bytes[1]};
    const cuuint32_t bx[3] = {box[0], box[1], box[2]};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&t->map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), d, st, bx, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    t->valid = (r == CUDA_SUCCESS);
    return t->valid;
}

bool nm_blur_uses_strip(const NmBlurArgs& a, const NmBlurTma* tma) { return strip_eligible(a, tma); }

bool nm_blur_make_tma(NmBlurTma* t, const float* src, int w, int h, int pitch, long long fstride,
                      int batch, int radius, bool words_u32)
{
    const CUtensorMapDataType dtype = words_u32 ? CU_TENSOR_MAP_DATA_TYPE_UINT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
    t->valid = t->valid_strip = t->valid_stream = false;
    if (radius < 1 || radius > 16 || w <= 0 || h <= 0 || batch <= 0) return false;
    if ((reinterpret_cast<uintptr_t>(src) & 15) || (pitch & 3) || (batch > 1 && (fstride & 3))) return false;
    EncodeTiledFn enc = get_encoder();
    if (!enc) return false;
    const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch * 4, (cuuint64_t)(batch > 1 ? fstride : (long long)pitch * h) * 4};
    const cuuint32_t box[3] = {(cuuint32_t)in_pitch(radius), (cuuint32_t)(kTH + 2 * radius), 1};
    const cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(&t->map, dtype, 3, const_cast<float*>(src), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    t->valid = (r == CUDA_SUCCESS);
    if (t->valid) {
        const cuuint32_t box_strip[3] = {(cuuint32_t)in_pitch(radius), (cuuint32_t)kCH, 1};
        r = enc(&t->map_strip, dtype, 3, const_cast<float*>(src), dims, strides, box_strip, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        t->valid_strip = (r == CUDA_SUCCESS);
        const cuuint32_t box_stream[3] = {(cuuint32_t)in_pitch(radius), (cuuint32_t)kGR, 1};
        r = enc(&t->map_stream, dtype, 3, const_cast<float*>(src), dims, strides, box_stream, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        t->valid_stream = (r == CUDA_SUCCESS);
    }
    return t->valid;
}

int nm_blur_launch(const NmBlurArgs& a, cudaStream_t stream, const NmBlurTma* tma)
{
    if (a.w <= 0 || a.h <= 0 || a.batch <= 0 || a.radius < 0 || a.radius > 45) return NM_ERR_INVALID;
    switch (a.radius) {
#define NM_CASE(R) case R: return launch_tile<R>(a, stream, tma);
        NM_CASE(1) NM_CASE(2) NM_CASE(3) NM_CASE(4) NM_CASE(5) NM_CASE(6) NM_CASE(7) NM_CASE(8)
        NM_CASE(9) NM_CASE(10) NM_CASE(11) NM_CASE(12) NM_CASE(13) NM_CASE(14) NM_CASE(15) NM_CASE(16)
#undef NM_CASE
        default: break;
    }
    if (a.scratch == nullptr) return NM_ERR_INVALID;
    dim3 grid(nm_div_up(a.w, 128), a.h, a.batch);
    blur_rows_generic<<<grid, 128, 0, stream>>>(a);
    NM_LAUNCH_CHECK();
    NmBlurArgs b = a;
    blur_cols_generic<<<grid, 128, 0, stream>>>(b);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_downsample_launch(float* dst, int dw, int dh, int dpitch, long long dfstride,
                         const float* src, int spitch, long long sfstride, int batch,
                         cudaStream_t stream)
{
    if (dw <= 0 || dh <= 0 || batch <= 0) return NM_ERR_INVALID;
    dim3 block(32, 8), grid(nm_div_up(dw, 32), nm_div_up(dh, 8), batch);
    downsample2_kernel<<<grid, block, 0, stream>>>(dst, dw, dh, dpitch, dfstride, src, spitch, sfstride);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

// Self-test of nm_gradient_from_diff against the library-routine expression (see nm_common.cuh).
namespace {
__device__ __forceinline__ unsigned st_hash(unsigned long long v)
{
    v ^= v >> 33; v *= 0xff51afd7ed558ccdULL; v ^= v >> 33; v *= 0xc4ceb9fe1a85ec53ULL; v ^= v >> 33;
    return (unsigned)v;
}
// argument generator: random sign; log-uniform magnitude over 2^-70 .. 2^66, or special patterns
__device__ __forceinline__ float st_value(unsigned h, unsigned mode)
{
    const float mant = 1.0f + (float)(h & 0x7fffff) * (1.0f / 8388608.0f);
    const int e = (int)((h >> 23) & 0xff) * 136 / 256 - 70;
    float v = ldexpf(mant, e);
    if (mode == 1) v = (float)((int)(h & 0x3ff) - 512) * 0.25f;         // quarter-integer pixel differences
    if (mode == 2) v = 0.0f;
    if (mode == 3) v = ldexpf(mant, (int)((h >> 23) & 0x1f) - 16);        // image-scale magnitudes 2^-16 .. 2^15
    if (mode == 4) v = ldexpf(mant, -140);                                // subnormal
    return (h >> 31) ? -v : v;
}
__global__ void gradient_selftest_kernel(long long n, unsigned seed, unsigned long long* mismatches)
{
    unsigned long long bad = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned h0 = st_hash(((unsigned long long)seed << 40) ^ (unsigned long long)i);
        const unsigned h1 = st_hash(((unsigned long long)seed << 40) ^ (unsigned long long)i ^ 0x9e3779b97f4a7c15ULL);
        const unsigned sel = st_hash(h0 ^ 0x5bd1e995u) & 31;
        // 0..7 wide range both, 8..19 image scale both, 20..23 quarter integers, 24/25 one zero,
        // 26/27 one subnormal, 28 wide x image scale, 29 both zero, 30 |dx| == |dy|, 31 image scale vs tiny
        unsigned my = sel < 8 ? 0 : sel < 20 ? 3 : sel < 24 ? 1 : sel == 24 ? 2 : sel == 26 ? 4 : sel == 29 ? 2 : 3;
        unsigned mxm = sel < 8 ? 0 : sel < 20 ? 3 : sel < 24 ? 1 : sel == 25 ? 2 : sel == 27 ? 4 : sel == 29 ? 2 : sel == 28 ? 0 : 3;
        float dy = st_value(h0, my), dx = st_value(h1, mxm);
        if (sel == 30) dx = (h1 & 1) ? dy : -dy;
        if (sel == 31) dx = ldexpf(dx, -70);
        const float2 a = nm_gradient_lib(dx, dy), b = nm_gradient_from_diff(dx, dy);
        if (__float_as_uint(a.x) != __float_as_uint(b.x) || __float_as_uint(a.y) != __float_as_uint(b.y)) ++bad;
    }
    if (bad) atomicAdd(mismatches, bad);
}
} // namespace

extern "C" int nm_selftest_gradient(long long n, unsigned seed, long long* mismatches_host)
{
    if (n <= 0 || !mismatches_host) return NM_ERR_INVALID;
    unsigned long long* d = nullptr;
    NM_CUDA_TRY(cudaMalloc(&d, sizeof(*d)));
    cudaMemset(d, 0, sizeof(*d));
    gradient_selftest_kernel<<<148 * 8, 256>>>(n, seed, d);
    cudaError_t e = cudaGetLastError();
    unsigned long long h = 0;
    if (e == cudaSuccess) e = cudaMemcpy(&h, d, sizeof(h), cudaMemcpyDeviceToHost);
    cudaFree(d);
    *mismatches_host = (long long)h;
    return nm_cuda_err(e);
}

// ---------------------------------------------------------------------------
// C-ABI
// ---------------------------------------------------------------------------
extern "C" int nm_blur_f32(float* result, const float* image, float* buffer, int width, int height,
                           const float* taps_dev, int radius, nm_stream_t stream)
{
    if (!result || !image || !taps_dev) return NM_ERR_INVALID;
    NmBlurArgs a{};
    a.src = image; a.dst = result; a.taps = taps_dev; a.dst2 = nullptr; a.scratch = buffer;
    a.w = width; a.h = height; a.src_pitch = width; a.dst_pitch = width; a.batch = 1; a.radius = radius;
    NmBlurTma tma;
    nm_blur_make_tma(&tma, image, width, height, width, 0, 1, radius);
    return nm_blur_launch(a, (cudaStream_t)stream, &tma);
}

extern "C" int nm_downsample2_f32(float* result, int rw, int rh, const float* source, int sw, int sh,
                                  nm_stream_t stream)
{
    if (!result || !source || 2 * (rw - 1) >= sw || 2 * (rh - 1) >= sh) return NM_ERR_INVALID;
    return nm_downsample_launch(result, rw, rh, rw, 0, source, sw, 0, 1, (cudaStream_t)stream);
}

extern "C" int nm_subtract_f32(const float* A, const float* B, float* C, int width, int height,
                               nm_stream_t stream)
{
    if (!A || !B || !C || width <= 0 || height <= 0) return NM_ERR_INVALID;
    const long long n = (long long)width * height;
    subtract_kernel<<<(unsigned)nm_div_up64(n, 256), 256, 0, (cudaStream_t)stream>>>(A, B, C, n);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

extern "C" int nm_gradient_f32(const float* source, float* grad2, int width, int height, nm_stream_t stream)
{
    if (!source || !grad2 || width <= 0 || height <= 0) return NM_ERR_INVALID;
    dim3 block(32, 8), grid(nm_div_up(width, 32), nm_div_up(height, 8));
    gradient_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(source, reinterpret_cast<float2*>(grad2), width, height);
    NM_LAUNCH_CHECK();
    return NM_OK;
}
