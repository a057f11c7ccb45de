// nm_orient_desc.cu -- dominant orientation and 128-D descriptor per keypoint.
//
// Replaces detect_orientations / kernel_orientations_optim (gpu/kernels/orientation.cu:
// 11-129, 219-230) and compute_sift_descriptors / kernel_descriptor_optim
// (gpu/kernels/descriptor.cu:32-145, 243-255) for the whole batch.
//
// Design: ONE WARP per keypoint (the reference spends a 484-thread and a 256-thread CTA
// per keypoint).  Histograms are privatised per lane in shared memory (bank = lane, no
// atomics, no float-atomic order nondeterminism -- the reference uses shared / global
// float atomics) and reduced across lanes in a fixed order with a swizzled read, so the
// output is bit-reproducible run to run.  All the reference's quirks that define its
// numbers are kept: positive-exponent Gaussian windows, the 10-pixel clamp of the
// orientation window, first-two-peaks-in-bin-order, first orientation only, diagonal-only
// 16x16 chunks of the descriptor window, no normalisation (SURVEY.md Q5,Q6,Q10,Q12,Q16).
#include "nm_sift_internal.cuh"
#include "nm_kpgeom.cuh"

namespace {

__device__ __forceinline__ float exp2f_approx(float x)
{
    float r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

constexpr int OR_WARPS = 8;      // warps per block, orientation
constexpr int NBINS = 36;
constexpr int OR_HP = 32;        // lane pitch of the private histograms (bank == lane)

__global__ void __launch_bounds__(OR_WARPS * 32) orient_kernel(const NmOctaveTable tab, int capacity,
                                                               const int* __restrict__ counts,
                                                               const float4* __restrict__ kpts,
                                                               const int* __restrict__ meta,
                                                               float2* __restrict__ orient)
{
    __shared__ float s_priv[OR_WARPS][NBINS * OR_HP];
    __shared__ float s_hist[OR_WARPS][NBINS + 4];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int f = blockIdx.y;
    const int j = blockIdx.x * OR_WARPS + wid;
    // count, payload and octave index are fetched together (slot j < capacity exists whatever the count): one memory
    // latency before the first gradient load instead of three dependent ones
    const long long kidx = (long long)f * capacity + j;
    const int n_kp = counts[f];
    const float4 kp = __ldg(kpts + kidx);
    const int oct = __ldg(meta + kidx);
    if (j >= n_kp) return;                                        // warp uniform
    float2 res = make_float2(-1.f, -1.f);                         // pyramidata.cu:90 fill
    if (!(kp.w < 0.f)) {                                          // orientation.cu:17
        const NmOctave& oc = tab.o[min(max(oct, 0), NM_MAX_OCTAVES - 1)];
        const KpGeom g = kp_geom(kp, oc.xper);
        float sigma_w;                                            // :26-30 (window clamped by the 22x22 block)
        const int W = kp_orient_radius(g, sigma_w);
        const float2* __restrict__ G = oc.grad + ((long long)f * 3 + g.level) * oc.level_elems +
                                       (long long)g.yi * oc.pitch + g.xi;      // at the keypoint; offsets below are 32-bit
        const int pitch = oc.pitch;
        float* priv = s_priv[wid];
        float* hist = s_hist[wid];
#pragma unroll
        for (int b = 0; b < NBINS; ++b) priv[b * OR_HP + lane] = 0.f;
        const int xmin = max(-W, -g.xi), xmax = min(W, oc.w - 1 - g.xi);   // :43-46
        const int ymin = max(-W, -g.yi), ymax = min(W, oc.h - 1 - g.yi);
        const int nx = xmax - xmin + 1, ny = ymax - ymin + 1;
        const int total = (nx > 0 && ny > 0) ? nx * ny : 0;
        const float den = __fmul_rn(sigma_w, __fadd_rn(sigma_w, sigma_w));  // 2*sigma_w*sigma_w
        // :56 exp(r2 / den) = 2^(r2 * log2(e) / den): one division per keypoint, ex2.approx per sample (2 ulp; the
        // orientation tolerance is 1e-3 rad, the measured deviation from the exact form stays below 1e-5)
        const float k_exp = __fdiv_rn(1.4426950408889634f, den);
        // :55 compares (double)r2 < W*W + 0.6; W*W + 0.6 is not an fp32 number, so for fp32 r2 that is
        // r2 < (the smallest fp32 above it)
        const float lim_f = __double2float_ru(__dadd_rn((double)(W * W), 0.6));
        // Window samples in raster order, 32 per step, four steps per round: the four gradient loads of a lane are issued
        // first (the maps of a batch live in HBM), then the four samples are accumulated.  Sample s sits at row s / nx,
        // column s % nx of the clipped window; nx <= 21 and s < 512, for which (s * ceil(2^16 / nx)) >> 16 is the exact
        // quotient -- no division and no carried position per sample.
        const int inv_nx = (65536 + max(nx, 1) - 1) / max(nx, 1);
        const float fx0 = (float)(xmin + g.xi), fy0 = (float)(ymin + g.yi);
        // The four loads of round k + 1 are issued before round k is accumulated (round 2 waited for its own loads: 18 % of
        // the warp samples sat on the first use of a gradient).
        auto load_round = [&](int s0, float2 (&gv)[4]) {
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const int sd = s0 + 32 * d;
                const int ryd = (sd * inv_nx) >> 16, rxd = sd - ryd * nx;
                gv[d] = make_float2(0.f, 0.f);
                if (sd < total) gv[d] = __ldg(G + ((ymin + ryd) * pitch + xmin + rxd));
            }
        };
        float2 gv[4];
        load_round(lane, gv);
        for (int s0 = lane; s0 < total; s0 += 128) {
            float2 gn[4];
            load_round(s0 + 128, gn);
#pragma unroll
            for (int d = 0; d < 4; ++d) {
                const int sd = s0 + 32 * d;
                const int ryd = (sd * inv_nx) >> 16, rxd = sd - ryd * nx;
                const float dx = __fsub_rn(__fadd_rn(fx0, (float)rxd), g.x);   // :52-53 (integers: the sums are exact)
                const float dy = __fsub_rn(__fadd_rn(fy0, (float)ryd), g.y);
                const float r2 = __fmaf_rn(dx, dx, __fmul_rn(dy, dy));         // :54
                if (sd < total && r2 < lim_f) {                               // :55
                    const float wgt = exp2f_approx(__fmul_rn(r2, k_exp));     // :56 (positive exponent)
                    // :57  bin = floor((float)((double)(36 theta) / 2 pi)).  The fp32 product v * (1 / 2 pi) is within
                    // 7e-6 of that quotient (v <= 227), so its floor is the reference's unless it lies within 1e-5
                    // of an integer; only then (2e-5 of the samples) the double division decides.
                    const float v36 = __fmul_rn(36.0f, gv[d].y);
                    const float qf = __fmul_rn(v36, 0.15915494309189535f);
                    float qfl = floorf(qf);
                    const float fr = __fsub_rn(qf, qfl);
                    if (!(fr > 1e-5f && fr < 0.99999f)) qfl = floorf((float)__ddiv_rn((double)v36, NM_TWO_PI_D));
                    int bin = (int)qfl;                               // theta in [0, 2 pi]: 0 .. 36
                    if ((unsigned)bin >= (unsigned)NBINS) { bin %= NBINS; if (bin < 0) bin += NBINS; }   // :58 bin % NBINS
                    float* p = priv + bin * OR_HP + lane;             // bank == lane: conflict free
                    *p = __fmaf_rn(gv[d].x, wgt, *p);                 // :58
                }
            }
#pragma unroll
            for (int d = 0; d < 4; ++d) gv[d] = gn[d];
        }
        __syncwarp();
        // fixed-order reduction: lane b owns bin b (and b+32 for lanes 0..3)
        for (int b = lane; b < NBINS; b += 32) {
            float acc = 0.f;
            const float* p = priv + b * OR_HP;
#pragma unroll 8
            for (int k = 0; k < 32; ++k) acc = __fadd_rn(acc, p[(k + lane) & 31]);   // rotated: conflict free
            hist[b] = acc;
        }
        __syncwarp();
        // 6x circular 3-tap box smoothing, Jacobi (intended semantics = orientation.cu:181-192)
        const int bm0 = (lane + NBINS - 1) % NBINS, bp0 = lane + 1;                    // neighbours of bin `lane` (< 32)
        const int b1 = lane + 32, bm1 = b1 - 1, bp1 = (b1 + 1) % NBINS;                // ... of bin `lane + 32` (lanes 0..3)
        for (int iter = 0; iter < 6; ++iter) {
            const float n0 = __fdiv_rn(__fadd_rn(__fadd_rn(hist[bm0], hist[lane]), hist[bp0]), 3.0f);
            float n1 = 0.f;
            if (lane < NBINS - 32) n1 = __fdiv_rn(__fadd_rn(__fadd_rn(hist[bm1], hist[b1]), hist[bp1]), 3.0f);
            __syncwarp();
            hist[lane] = n0;
            if (lane < NBINS - 32) hist[b1] = n1;
            __syncwarp();
        }
        float m = fmaxf(0.f, hist[lane]);                          // :93-95
        if (lane < NBINS - 32) m = fmaxf(m, hist[lane + 32]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, d));
        const float thr = (float)__dmul_rn((double)m, 0.8);        // :96
        float th0 = -1.f, th1 = -1.f;
        bool pk0 = false, pk1 = false;
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const int b = lane + 32 * half;
            if (b < NBINS) {
                const float h0 = hist[b], hm = hist[(b + NBINS - 1) % NBINS], hp = hist[(b + 1) % NBINS];
                if (h0 > thr && h0 > hm && h0 > hp) {              // :107
                    const double num = __dmul_rn(-0.5, (double)__fsub_rn(hp, hm));
                    const double dn = (double)__fsub_rn(__fadd_rn(hp, hm), __fmul_rn(2.0f, h0));
                    const float di = (float)__ddiv_rn(num, dn);    // :108
                    const float th = (float)__ddiv_rn(
                        __dmul_rn(NM_TWO_PI_D, __dadd_rn((double)__fadd_rn((float)b, di), 0.5)), 36.0);  // :109
                    if (half == 0) { pk0 = true; th0 = th; } else { pk1 = true; th1 = th; }
                }
            }
        }
        // first two peaks in ascending bin order (:116-128)
        const unsigned m0 = __ballot_sync(0xffffffffu, pk0);
        const unsigned m1 = __ballot_sync(0xffffffffu, pk1);
        float first = -1.f, second = -1.f;
        int found = 0;
        unsigned mm = m0;
        while (mm && found < 2) {
            const int src = __ffs(mm) - 1; mm &= mm - 1;
            const float v = __shfl_sync(0xffffffffu, th0, src);
            if (found == 0) first = v; else second = v;
            ++found;
        }
        mm = m1;
        while (mm && found < 2) {
            const int src = __ffs(mm) - 1; mm &= mm - 1;
            const float v = __shfl_sync(0xffffffffu, th1, src);
            if (found == 0) first = v; else second = v;
            ++found;
        }
        res = make_float2(first, second);
    }
    if (lane == 0) orient[kidx] = res;
}

// ------------------------------- descriptor -----------------------------------
constexpr int DE_WARPS = 4;
constexpr int DE_BINS = 128;
constexpr int DE_COPIES = 16;    // private histogram copies per warp (lanes l, l + 16 share one): 8 KB per keypoint
                                 // in flight instead of 16 -> twice the resident warps (the kernel is latency bound)

// Exact mode: the reference's mixed double/float expression shapes (descriptor.cu:98-115, with
// the DFMA contractions of its sm_100a SASS).  describe_fast_kernel below evaluates the same
// formulas in fp32 (the bins and trilinear weights are continuous in nx, ny, nt, so the fp32
// evaluation stays within ~1e-6 relative of the exact one; the tolerance is 1e-3, BASELINE.json).
__global__ void __launch_bounds__(DE_WARPS * 32) describe_kernel(const NmOctaveTable tab, int capacity,
                                                                 const int* __restrict__ counts,
                                                                 const float4* __restrict__ kpts,
                                                                 const int* __restrict__ meta,
                                                                 const float2* __restrict__ orient,
                                                                 float* __restrict__ desc, float* __restrict__ xo,
                                                                 float* __restrict__ yo, int num_dogs)
{
    extern __shared__ __align__(16) float s_h[];      // [DE_WARPS][128 bins][DE_COPIES private copies]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int f = blockIdx.y;
    const int j = blockIdx.x * DE_WARPS + wid;
    if (j >= counts[f]) return;                                   // warp uniform
    const long long kidx = (long long)f * capacity + j;
    const float4 kp = kpts[kidx];
    const NmOctave& oc = tab.o[meta[kidx]];
    const KpGeom g = kp_geom(kp, oc.xper);                        // descriptor.cu:41-47
    float* dout = desc + kidx * DE_BINS;
    if (g.xi < 0 || g.xi >= oc.w || g.yi < 0 || g.yi >= oc.h || g.level < 0 || g.level >= num_dogs)
        return;                                                   // :49 (slot left as is)
    float* hist = s_h + wid * (DE_BINS * DE_COPIES);
#pragma unroll 4
    for (int b = 0; b < DE_BINS * DE_COPIES / 32; ++b) hist[b * 32 + lane] = 0.f;
    __syncwarp();

    const KpDescWindow dw = kp_desc_window(g, oc.w, oc.h);                               // :54-65
    const float SBP = dw.SBP;
    const int xmin = dw.xmin, xmax = dw.xmax, ymin = dw.ymin, ymax = dw.ymax, chunks = dw.chunks;
    const float th0 = orient[kidx].x;                                                    // :89; in [0, 2 pi] or -1 (no peak),
                                                                                         // so gradient angle - th0 is in (-2 pi, 2 pi + 1]
    const float st0f = sinf(th0), ct0f = cosf(th0);                                      // :90-91 (float overloads)
    const double st0 = (double)st0f, ct0 = (double)ct0f;
    const float2* __restrict__ G = oc.grad + ((long long)f * 3 + g.level) * oc.level_elems +
                                   (long long)g.yi * oc.pitch + g.xi;
    const int total = chunks * 256;
    // The gradient samples come from HBM (the maps of a 64-frame batch are 4.5 GB, L2 hit rate 23 %)
    // and only ~11 warps fit an SM next to the private histograms, so the load of iteration i+1 is
    // issued before the arithmetic of iteration i (ncu: 53 % of the stall samples sat on the first
    // use of the loaded value).
    auto sample_pos = [&](int s, int& cx, int& cy) -> bool {
        const int c = s >> 8, ty = (s >> 4) & 15, tx = s & 15;
        cx = xmin + tx + 16 * c; cy = ymin + ty + 16 * c;         // diagonal chunks only (:142-143)
        return s < total && cx <= xmax && cy <= ymax;             // :96
    };
    // one sample: rotate into the keypoint frame, weight, spread into the 2 x 2 x 2 neighbouring bins
    auto process = [&](const int cx, const int cy, const float2 gv, const bool act) {
        const float mod = gv.x;
        const float dx = __fsub_rn((float)(g.xi + cx), g.x);          // :102-103
        const float dy = __fsub_rn((float)(g.yi + cy), g.y);
        const float theta = nm_mod_2pi_once(__fsub_rn(gv.y, th0));                                             // :100
        const float nx = (float)__ddiv_rn(__fma_rn(ct0, (double)dx, __dmul_rn(st0, (double)dy)), (double)SBP);  // :104
        const float ny = (float)__ddiv_rn(__fma_rn(ct0, (double)dy, -__dmul_rn(st0, (double)dx)), (double)SBP); // :105
        const float nt = (float)__ddiv_rn((double)__fmul_rn(8.0f, theta), NM_TWO_PI_D);                         // :107
        const float win = (float)exp(__dmul_rn((double)__fmaf_rn(nx, nx, __fmul_rn(ny, ny)), 0.125));           // :108
        const int binx = (int)floor(__dadd_rn((double)nx, -0.5));                                               // :110
        const int biny = (int)floor(__dadd_rn((double)ny, -0.5));
        const float rbinx = (float)__dsub_rn((double)nx, __dadd_rn((double)binx, 0.5));                         // :113
        const float rbiny = (float)__dsub_rn((double)ny, __dadd_rn((double)biny, 0.5));
        const int bint = (int)floorf(nt);                             // :112
        const float rbint = __fsub_rn(nt, (float)bint);               // :115
        const float wm = __fmul_rn(win, mod);                         // :128-129 (left to right)
        // the 2 x 2 x 2 neighbouring bins (:118-137).  Same products in the same order as the
        // reference (((win*mod)*wx)*wy)*wt; the bin addresses are two base pointers (orientation
        // bins bint, bint+1 of cell (biny, binx)) plus compile-time cell offsets, instead of a
        // recomputed index per contribution (integer/address work was a third of the kernel).
        const int bx0 = binx + 2, by0 = biny + 2;
        const bool vx0 = (unsigned)bx0 < 4u, vx1 = (unsigned)(bx0 + 1) < 4u;       // :122-125
        const bool vy0 = (unsigned)by0 < 4u, vy1 = (unsigned)(by0 + 1) < 4u;
        float* hp = hist + (lane & (DE_COPIES - 1)) + (by0 * 32 + bx0 * 8) * DE_COPIES;   // only dereferenced for valid cells
        float* h0 = hp + (bint & 7) * DE_COPIES;                      // :133 (bint + dbt) % 8
        float* h1 = hp + ((bint + 1) & 7) * DE_COPIES;
        const float ax0 = fabsf(__fsub_rn(1.f, rbinx)), ax1 = fabsf(__fsub_rn(0.f, rbinx));
        const float ay0 = fabsf(__fsub_rn(1.f, rbiny)), ay1 = fabsf(__fsub_rn(0.f, rbiny));
        const float at0 = fabsf(__fsub_rn(1.f, rbint)), at1 = fabsf(__fsub_rn(0.f, rbint));
        const float a0 = __fmul_rn(wm, ax0), a1 = __fmul_rn(wm, ax1);
        constexpr int OX = 8 * DE_COPIES, OY = 32 * DE_COPIES;        // next cell in x / y (floats)
        // lanes l and l + 16 share a private copy: the two half-warps update one after the other
        // (computing the eight contributions once, outside the phases, measured slower: 2.27 -> 2.61 ms)
#pragma unroll
        for (int ph = 0; ph < 32 / DE_COPIES; ++ph) {
        if (act && (lane / DE_COPIES) == ph) {
        if (vx0 && vy0) {
            const float w = __fmul_rn(a0, ay0);
            h0[0] = __fadd_rn(h0[0], __fmul_rn(w, at0)); h1[0] = __fadd_rn(h1[0], __fmul_rn(w, at1));   // :135
        }
        if (vx0 && vy1) {
            const float w = __fmul_rn(a0, ay1);
            h0[OY] = __fadd_rn(h0[OY], __fmul_rn(w, at0)); h1[OY] = __fadd_rn(h1[OY], __fmul_rn(w, at1));
        }
        if (vx1 && vy0) {
            const float w = __fmul_rn(a1, ay0);
            h0[OX] = __fadd_rn(h0[OX], __fmul_rn(w, at0)); h1[OX] = __fadd_rn(h1[OX], __fmul_rn(w, at1));
        }
        if (vx1 && vy1) {
            const float w = __fmul_rn(a1, ay1);
            h0[OX + OY] = __fadd_rn(h0[OX + OY], __fmul_rn(w, at0)); h1[OX + OY] = __fadd_rn(h1[OX + OY], __fmul_rn(w, at1));
        }
        }
        __syncwarp();
        }
    };
    // DEPTH gradient loads stay in flight per lane (DRAM latency ~1 us against ~150 instructions per
    // sample and under 3 resident warps per scheduler)
    constexpr int DEPTH = 4;
    const int dpitch = oc.pitch;               // offsets inside one level fit 32 bits
    int pcx[DEPTH], pcy[DEPTH];
    bool pv[DEPTH];
    float2 pg[DEPTH];
#pragma unroll
    for (int d = 0; d < DEPTH; ++d) {
        pv[d] = sample_pos(lane + 32 * d, pcx[d], pcy[d]);
        pg[d] = make_float2(0.f, 0.f);
        if (pv[d]) pg[d] = __ldg(G + (pcy[d] * dpitch + pcx[d]));
    }
    for (int s = lane; s < total; s += 32 * DEPTH) {
#pragma unroll
        for (int d = 0; d < DEPTH; ++d) {
            const int cx = pcx[d], cy = pcy[d];
            const bool valid = pv[d];
            const float2 gv = pg[d];
            pv[d] = sample_pos(s + 32 * (d + DEPTH), pcx[d], pcy[d]);
            if (pv[d]) pg[d] = __ldg(G + (pcy[d] * dpitch + pcx[d]));
            process(cx, cy, gv, valid);
        }
    }
    __syncwarp();
    // fixed-order reduction; lane owns bins lane, lane+32, lane+64, lane+96
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int b = lane + 32 * q;
        float acc = 0.f;
#pragma unroll 8
        for (int k = 0; k < DE_COPIES; ++k)
            acc = __fadd_rn(acc, hist[b * DE_COPIES + ((k + lane / (32 / DE_COPIES)) & (DE_COPIES - 1))]);   // rotated: conflict free
        dout[b] = acc;
    }
    if (lane == 0) { xo[kidx] = kp.x; yo[kidx] = kp.y; }              // :76
}

// ------------------------------- descriptor, fp32 mode -----------------------------------
// The descriptor formulas in fp32, arranged for a low instruction count per sample (the kernel is issue bound: the
// round-1 fp32 kernel, which walked the window one flat sample index at a time, took 135 warp instructions per 32
// samples, 5 350 per keypoint):
//   * the window is walked chunk by chunk and row by row (lane = column (0..15) + 16 * (row & 1), eight row steps
//     per 16 x 16 chunk), so sample positions, validity and gradient addresses are increments, not a decode of a
//     flat sample index; the eight gradient loads of the NEXT chunk are issued before the current chunk's
//     arithmetic;
//   * the rotation into the keypoint frame is folded with the 1 / SBP scale: nx = sn * dy + (cs * dx), one FFMA per
//     coordinate with the per-chunk terms hoisted;
//   * exp(r2 / 8) through ex2.approx (2 ulp; the tolerance is 1e-3), contributions added with one FFMA each.
// Reduction order over the copies is fixed, so the output is bit-reproducible run to run.
// Variants measured on a B200 with 64 x 1080p frames, against this kernel's 1.54 ms: the round-1 kernel 2.26 ms;
// without the skip of sample rows that have no active lane 1.63; two passes of 16 lanes instead of the split by bin
// parity 1.87; a test of the row against ymax before the sample arithmetic 1.60; packed fp32 pairs (FFMA2) for the
// sample arithmetic 1.71 (1.84 without the row skip); 32 histogram copies, one per lane, 1.97 (2.03 packed, 1.96 in
// two-warp CTAs); register caps for 6 / 7 CTAs per SM 1.88 - 2.28.
__global__ void __launch_bounds__(DE_WARPS * 32) describe_fast_kernel(const NmOctaveTable tab, int capacity,
                                                                     const int* __restrict__ counts,
                                                                     const float4* __restrict__ kpts,
                                                                     const int* __restrict__ meta,
                                                                     const float2* __restrict__ orient,
                                                                     float* __restrict__ desc, float* __restrict__ xo,
                                                                     float* __restrict__ yo, int num_dogs)
{
    extern __shared__ __align__(16) float s_h[];      // [DE_WARPS][128 bins][DE_COPIES]
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int f = blockIdx.y;
    const int j = blockIdx.x * DE_WARPS + wid;
    const long long kidx = (long long)f * capacity + j;
    const int n_kp = counts[f];                                   // fetched together with the slot's payload (see orient_kernel)
    const float4 kp = __ldg(kpts + kidx);
    const int oct = __ldg(meta + kidx);
    const float2 ori = __ldg(orient + kidx);
    if (j >= n_kp) return;                                        // warp uniform
    const NmOctave& oc = tab.o[min(max(oct, 0), NM_MAX_OCTAVES - 1)];
    const KpGeom g = kp_geom(kp, oc.xper);                        // descriptor.cu:41-47
    float* dout = desc + kidx * DE_BINS;
    if (g.xi < 0 || g.xi >= oc.w || g.yi < 0 || g.yi >= oc.h || g.level < 0 || g.level >= num_dogs)
        return;                                                   // :49 (slot left as is)
    float* hist = s_h + wid * (DE_BINS * DE_COPIES);
    {
        float4* h4 = reinterpret_cast<float4*>(hist);
#pragma unroll
        for (int b = 0; b < DE_BINS * DE_COPIES / 128; ++b) h4[b * 32 + lane] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncwarp();

    const KpDescWindow dw = kp_desc_window(g, oc.w, oc.h);        // :54-65
    const int xmin = dw.xmin, xmax = dw.xmax, ymin = dw.ymin, ymax = dw.ymax, chunks = dw.chunks;
    const float th0 = ori.x;                                      // :89; in [0, 2 pi] or -1 (no peak)
    const float inv_sbp = __fdiv_rn(1.0f, dw.SBP);
    const float cs = __fmul_rn(cosf(th0), inv_sbp), sn = __fmul_rn(sinf(th0), inv_sbp);   // :90-91 folded with 1 / SBP (:104-105)
    const int pitch = oc.pitch;
    const float2* __restrict__ G = oc.grad + ((long long)f * 3 + g.level) * oc.level_elems +
                                   (long long)g.yi * pitch + g.xi;             // offsets inside one level fit 32 bits
    float* const hcopy = hist + (lane & (DE_COPIES - 1));
    const int tx = lane & 15, ty = lane >> 4;

    // gradient samples of chunk c for this lane: column xmin + 16 c + tx, rows ymin + 16 c + ty + 2 i (:94-97, :142-143)
    auto load_chunk = [&](int c, float2 (&gv)[8]) {
        const int bx = xmin + 16 * c + tx, by = ymin + 16 * c + ty;
        const float2* p = G + (by * pitch + bx);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            gv[i] = make_float2(0.f, 0.f);
            if (c < chunks && bx <= xmax && by + 2 * i <= ymax) gv[i] = __ldg(p + 2 * i * pitch);
        }
    };
    auto process_chunk = [&](int c, const float2 (&cur)[8]) {
        const int bx = xmin + 16 * c + tx, by = ymin + 16 * c + ty;
        const bool vx = bx <= xmax;
        const float dx = __fsub_rn((float)(g.xi + bx), g.x);                   // :102
        const float ax = __fmul_rn(cs, dx), ay = -__fmul_rn(sn, dx);
        const float fy0 = (float)(g.yi + by);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float dy = __fsub_rn(__fadd_rn(fy0, (float)(2 * i)), g.y);   // :103 (integers: the sum is exact)
            const float nx = __fmaf_rn(sn, dy, ax), ny = __fmaf_rn(cs, dy, ay);            // :104-105
            const float fx = floorf(__fsub_rn(nx, 0.5f)), fy = floorf(__fsub_rn(ny, 0.5f));   // :110-111
            const int bx0 = (int)fx + 2, by0 = (int)fy + 2;
            // about a third of the window (corners outside the rotated 4 x 4 cell grid) lands in no bin (:122-125)
            const bool act = vx && by + 2 * i <= ymax && (unsigned)(bx0 + 1) <= 4u && (unsigned)(by0 + 1) <= 4u;
            // rows of the chunk in which no lane lands in a cell (below the window, or the chunk's corner outside the
            // rotated grid) are about four in ten: the weights and the two histogram passes are skipped for them
            if (!__any_sync(0xffffffffu, act)) continue;
            const float theta = nm_mod_2pi_once(__fsub_rn(cur[i].y, th0));     // :100
            const float nt = __fmul_rn(theta, 1.2732395447351628f);            // :107, 8 / (2 pi)
            const float ft = floorf(nt);
            const int bint = (int)ft;                                          // :112
            const float rbint = __fsub_rn(nt, ft);                             // :115
            const float r2 = __fmaf_rn(nx, nx, __fmul_rn(ny, ny));
            const float win = exp2f_approx(__fmul_rn(r2, 0.18033688011112042f));   // :108  exp(r2 / 8) = 2^(r2 * log2(e) / 8)
            const float rbinx = __fsub_rn(nx, __fadd_rn(fx, 0.5f)), rbiny = __fsub_rn(ny, __fadd_rn(fy, 0.5f));   // :113-114
            const float wm = __fmul_rn(win, cur[i].x);                         // :128-129
            const float a1 = __fmul_rn(wm, rbinx), a0 = __fsub_rn(wm, a1);     // wm * |1 - rbinx|, wm * |rbinx|
            const float w01 = __fmul_rn(a0, rbiny), w00 = __fsub_rn(a0, w01);
            const float w11 = __fmul_rn(a1, rbiny), w10 = __fsub_rn(a1, w11);
            const float at1 = rbint, at0 = __fsub_rn(1.f, rbint);
            float* hp = hcopy + (by0 * 32 + bx0 * 8) * DE_COPIES;                 // only dereferenced for valid cells
            float* h0 = hp + (bint & 7) * DE_COPIES;                              // :133 (bint + dbt) % 8
            float* h1 = hp + ((bint + 1) & 7) * DE_COPIES;
            constexpr int OX = 8 * DE_COPIES, OY = 32 * DE_COPIES;
            const bool vx0 = (unsigned)bx0 < 4u, vx1 = (unsigned)(bx0 + 1) < 4u;            // :122-125
            const bool vy0 = (unsigned)by0 < 4u, vy1 = (unsigned)(by0 + 1) < 4u;
            // The eight bins of a sample are distinct addresses: all eight loads are issued before the first store, so a
            // sample costs ONE shared-memory round trip (load -> FFMA -> store) instead of eight dependent ones -- the
            // compiler cannot know that h0[...] and h1[...] never alias and would order every load after the previous
            // store (the round-1 kernel was bound by exactly that chain: twice the histogram copies, i.e. half the
            // resident warps, made it 2.3x slower).
            const bool p00 = vx0 && vy0, p01 = vx0 && vy1, p10 = vx1 && vy0, p11 = vx1 && vy1;
            // Lanes l and l + 16 share a copy.  A sample's two orientation bins have different parities, so in the first
            // pass every lane adds to the bin whose parity is its half-warp's and in the second to the other one: the two
            // lanes of a copy never meet in a pass, all 32 lanes work in both (round 2 had two passes of 16 lanes with all
            // eight bins each), and with bank = copy + 16 * (bin & 1) each of the four accesses of a pass is conflict free.
            const bool sw = ((bint ^ (lane >> 4)) & 1) != 0;
            float* pa = sw ? h1 : h0;
            float* pb = sw ? h0 : h1;
            const float ta = sw ? at1 : at0, tb = sw ? at0 : at1;
#pragma unroll
            for (int ph = 0; ph < 2; ++ph) {
                float* q = ph ? pb : pa;
                const float tq = ph ? tb : ta;
                if (act) {
                    float v0 = 0.f, v1 = 0.f, v2 = 0.f, v3 = 0.f;
                    if (p00) v0 = q[0];
                    if (p01) v1 = q[OY];
                    if (p10) v2 = q[OX];
                    if (p11) v3 = q[OX + OY];
                    v0 = __fmaf_rn(w00, tq, v0); v1 = __fmaf_rn(w01, tq, v1);                                            // :135
                    v2 = __fmaf_rn(w10, tq, v2); v3 = __fmaf_rn(w11, tq, v3);
                    if (p00) q[0] = v0;
                    if (p01) q[OY] = v1;
                    if (p10) q[OX] = v2;
                    if (p11) q[OX + OY] = v3;
                }
                __syncwarp();
            }
        }
    };
    // the loads of chunk c + 1 are in flight while chunk c is accumulated (a two-register-set ping-pong, an early exit
    // for the rows below the window and a register cap for 5 CTAs / SM were each measured slower: 1.86 -> 2.24 ms)
    float2 cur[8], nxt[8];
    load_chunk(0, cur);
    for (int c = 0; c < chunks; ++c) {
        load_chunk(c + 1, nxt);
        process_chunk(c, cur);
#pragma unroll
        for (int i = 0; i < 8; ++i) cur[i] = nxt[i];
    }
    __syncwarp();
    // fixed-order reduction; lane owns bins lane, lane+32, lane+64, lane+96
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int b = lane + 32 * q;
        float acc = 0.f;
#pragma unroll 8
        for (int k = 0; k < DE_COPIES; ++k)
            acc = __fadd_rn(acc, hist[b * DE_COPIES + ((k + lane / (32 / DE_COPIES)) & (DE_COPIES - 1))]);   // rotated: conflict free
        dout[b] = acc;
    }
    if (lane == 0) { xo[kidx] = kp.x; yo[kidx] = kp.y; }              // :76
}

// ---------------------- compat: flat keypoint lists (one octave) ----------------------
__global__ void compat_fill_meta(int* meta, int* count, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) meta[i] = 0;
    if (i == 0) *count = n;
}

} // namespace

int nm_orient_launch(const NmOctaveTable& tab, int batch, int capacity, const int* counts,
                     const float4* kpts, const int* meta, float2* orient, cudaStream_t stream)
{
    dim3 grid(nm_div_up(capacity, OR_WARPS), batch);
    orient_kernel<<<grid, OR_WARPS * 32, 0, stream>>>(tab, capacity, counts, kpts, meta, orient);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

int nm_describe_launch(const NmOctaveTable& tab, int batch, int capacity, const int* counts,
                       const float4* kpts, const int* meta, const float2* orient, float* desc,
                       float* x, float* y, int num_dogs, int exact, cudaStream_t stream)
{
    static NmDeviceOnce once;
    constexpr int smem = DE_WARPS * DE_BINS * DE_COPIES * (int)sizeof(float);
    if (once.first()) {
        NM_CUDA_TRY(cudaFuncSetAttribute(describe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        NM_CUDA_TRY(cudaFuncSetAttribute(describe_fast_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        once.done();
    }
    const auto kernel = exact ? describe_kernel : describe_fast_kernel;
    dim3 grid(nm_div_up(capacity, DE_WARPS), batch);
    kernel<<<grid, DE_WARPS * 32, smem, stream>>>(tab, capacity, counts, kpts, meta, orient, desc, x, y, num_dogs);
    NM_LAUNCH_CHECK();
    return NM_OK;
}

// ---------------------------------------------------------------------------
// C-ABI (compat granularity): one octave, flat keypoint list, dense gradient maps
// laid out like PyramidData::_grad (level * oh*ow + y*ow + x).
// ---------------------------------------------------------------------------
static int compat_table(NmOctaveTable& tab, const float* grad2, int ow, int oh, float xper)
{
    tab.n_oct = 1;
    NmOctave& oc = tab.o[0];
    oc.levels = nullptr; oc.bitmap = nullptr; oc.wprefix = nullptr; oc.need = nullptr; oc.cand_n = nullptr; oc.cand = nullptr;
    oc.grad = reinterpret_cast<float2*>(const_cast<float*>(grad2));
    oc.w = ow; oc.h = oh; oc.pitch = ow; oc.wpr = nm_div_up(ow, 32);
    oc.level_elems = (long long)ow * oh;
    oc.xper = xper;
    return NM_OK;
}

namespace {
struct CompatScratch { int* counts; int* meta; };
int compat_scratch(CompatScratch& sc, int n, cudaStream_t st)
{
    NM_CUDA_TRY(nm_ws_alloc(&sc.counts, sizeof(int), st));
    NM_CUDA_TRY(nm_ws_alloc(&sc.meta, sizeof(int) * n, st));
    compat_fill_meta<<<nm_div_up(n, 256), 256, 0, st>>>(sc.meta, sc.counts, n);
    NM_LAUNCH_CHECK();
    return NM_OK;
}
} // namespace

extern "C" int nm_orientations_f32(const float* kpts4, const float* grad2, int num_pts, int octave_width,
                                   int octave_height, float gauss_factor, float xper, float* result2,
                                   nm_stream_t stream)
{
    if (!kpts4 || !grad2 || !result2 || num_pts <= 0 || octave_width <= 0 || octave_height <= 0) return NM_ERR_INVALID;
    if (gauss_factor != 1.5f) return NM_ERR_UNSUPPORTED;   // the reference hard-codes 1.5f (siftfunctions.cu:150)
    cudaStream_t st = (cudaStream_t)stream;
    NmOctaveTable tab; compat_table(tab, grad2, octave_width, octave_height, xper);
    CompatScratch sc{};
    int rc = compat_scratch(sc, num_pts, st);
    if (rc == NM_OK)
        rc = nm_orient_launch(tab, 1, num_pts, sc.counts, reinterpret_cast<const float4*>(kpts4), sc.meta,
                              reinterpret_cast<float2*>(result2), st);
    if (sc.counts) cudaFreeAsync(sc.counts, st);
    if (sc.meta) cudaFreeAsync(sc.meta, st);
    return rc;
}

extern "C" int nm_descriptors_f32(const float* kpts4, const float* orient2, const float* grad2, int num_pts,
                                  int octave_width, int octave_height, int num_dogs, float xper,
                                  float* desc, float* x, float* y, nm_stream_t stream)
{
    if (!kpts4 || !orient2 || !grad2 || !desc || !x || !y || num_pts <= 0 || octave_width <= 0 || octave_height <= 0)
        return NM_ERR_INVALID;
    cudaStream_t st = (cudaStream_t)stream;
    NmOctaveTable tab; compat_table(tab, grad2, octave_width, octave_height, xper);
    CompatScratch sc{};
    int rc = compat_scratch(sc, num_pts, st);
    if (rc == NM_OK)
        rc = nm_describe_launch(tab, 1, num_pts, sc.counts, reinterpret_cast<const float4*>(kpts4), sc.meta,
                                reinterpret_cast<const float2*>(orient2), desc, x, y, num_dogs, 0, st);
    if (sc.counts) cudaFreeAsync(sc.counts, st);
    if (sc.meta) cudaFreeAsync(sc.meta, st);
    return rc;
}
