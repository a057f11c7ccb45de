// nm_chain.cuh -- the chaining rule of a registered frame stream, shared by the mosaic placement (place_kernel,
// nm_mosaic.cu) and the initial poses of the chain adjustment (nm_ransac_adjust_chain_f32, nm_ransac.cu), so that both
// turn a pairwise model into the same step.
#pragma once
#include "nm_common.cuh"

__device__ __forceinline__ double nm_det3d(const double* a)
{
    return a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6]);
}
// r = a^-1 (adjugate over the determinant)
__device__ __forceinline__ void nm_inv3d(const double* a, double det, double* r)
{
    r[0] = (a[4] * a[8] - a[5] * a[7]) / det;
    r[1] = (a[2] * a[7] - a[1] * a[8]) / det;
    r[2] = (a[1] * a[5] - a[2] * a[4]) / det;
    r[3] = (a[5] * a[6] - a[3] * a[8]) / det;
    r[4] = (a[0] * a[8] - a[2] * a[6]) / det;
    r[5] = (a[2] * a[3] - a[0] * a[5]) / det;
    r[6] = (a[3] * a[7] - a[4] * a[6]) / det;
    r[7] = (a[1] * a[6] - a[0] * a[7]) / det;
    r[8] = (a[0] * a[4] - a[1] * a[3]) / det;
}
__device__ __forceinline__ double nm_max_abs9(const double* a)
{
    double m = 0.0;
    for (int i = 0; i < 9; ++i) m = fmax(m, fabs(a[i]));
    return m;
}

// divide by the power of two at the largest absolute entry (max in [0.5, 1) afterwards): exact, so a chain of
// thousands of frames neither overflows nor picks up rounding from the rescaling
__device__ __forceinline__ void nm_renormalise(double* a)
{
    const double m = nm_max_abs9(a);
    if (!(m > 0.0) || !isfinite(m)) return;
    int e;
    frexp(m, &e);
    const double s = ldexp(1.0, -e);
    for (int i = 0; i < 9; ++i) a[i] *= s;
}

// The step of one pair (model H: frame p -> frame p + 1, fp32, row-major): r = H^-1 in fp64, or the identity when
// `ok` is false or H is non-finite or singular (|det| <= 1e-12 max|H|^3).  Returns whether H was inverted.
__device__ __forceinline__ bool nm_chain_step(const float* H, bool ok, double* r)
{
    double h[9];
    for (int i = 0; i < 9; ++i) { h[i] = (double)H[i]; ok = ok && isfinite(h[i]); }
    if (ok) {
        const double m = nm_max_abs9(h), det = nm_det3d(h);
        ok = fabs(det) > 1e-12 * m * m * m;
        if (ok) nm_inv3d(h, det, r);
    }
    if (!ok) for (int i = 0; i < 9; ++i) r[i] = (i % 4 == 0) ? 1.0 : 0.0;
    return ok;
}
