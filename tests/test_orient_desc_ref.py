"""The float64 / IEEE restatement of the orientation and descriptor semantics (tests/orient_desc_ref.py) against the
CPU oracle's orc_orientations / orc_descriptors.  No GPU: this proves the restatement that
tests/test_gpu_orient_desc_rules.py holds the CUDA kernels to.

Bounds.  The oracle sums a bin's weighted samples in raster order in fp32 (at most 441 positive terms), with expf
weights (< 2 ulp) and 18 fp32 operations of smoothing per bin; the restatement sums in float64 and rounds once.  So
the two smoothed histograms differ by a relative perturbation below 500 * 2^-24 < 2^-15 = ORACLE_EPS: peak decisions
must agree wherever the restatement's margin exceeds it, and an angle may move by sens * ORACLE_EPS plus 1e-6 rad
for the fp32 roundings of the fit (2 ulp of 2 pi).  The oracle's descriptor arithmetic is within 2^-20.8 of float64
per sample relative to win * mod (measured on impulses below) and a descriptor entry sums positive contributions, so
an entry is held to 2^-20 * wm."""
import fractions

import numpy as np
import pytest

from tests import orient_desc_ref as R
from tests._util import ang_diff, orc_descriptors, orc_orientations

ORACLE_EPS = 2.0 ** -15
FIT_ULPS = 1e-6
ORACLE_DESC = 2.0 ** -20


@pytest.fixture(scope="module")
def lib(oracle):
    return oracle.lib


def _ulp_exact_fmaf(a, b, c):
    """fmaf through exact rational arithmetic: the float32 nearest to a * b + c, ties to even."""
    out = np.empty(len(a), np.float32)
    for i, (x, y, z) in enumerate(zip(a, b, c)):
        e = fractions.Fraction(float(x)) * fractions.Fraction(float(y)) + fractions.Fraction(float(z))
        f = np.float32(float(e))
        cands = [np.nextafter(f, np.float32(-np.inf)), f, np.nextafter(f, np.float32(np.inf))]
        d = [abs(fractions.Fraction(float(v)) - e) for v in cands]
        best = min(d)
        ties = [v for v, dv in zip(cands, d) if dv == best]
        out[i] = ties[0] if len(ties) == 1 else next(v for v in ties if not (v.view(np.int32) & 1))
    return out


def test_fmaf_is_correctly_rounded():
    """Random operands, and a * b + c = 1 + 2^-24 + 2^-70 (8392705 * 16769026 = 2^47 + 2): the double sum is the
    midpoint 1 + 2^-24 of two floats, the exact value lies above it and rounds up, where a second rounding of the
    double sum would round to even, down to 1."""
    rng = np.random.default_rng(5)
    a = (rng.standard_normal(4000) * 10).astype(np.float32)
    b = (rng.standard_normal(4000) * 10).astype(np.float32)
    c = (rng.standard_normal(4000) * 100).astype(np.float32)
    a = np.append(a, [8392705 * 2.0 ** -35, 8392705 * 2.0 ** -35]).astype(np.float32)
    b = np.append(b, [16769026 * 2.0 ** -36, -16769026 * 2.0 ** -36]).astype(np.float32)
    c = np.append(c, [1.0, 1.0]).astype(np.float32)
    got = R.fmaf(a, b, c)
    assert got[-2] == np.float32(1 + 2.0 ** -23) and got[-1] == np.float32(1 - 2.0 ** -24)
    assert np.array_equal(got.view(np.int32), _ulp_exact_fmaf(a, b, c).view(np.int32))


def test_impulse_orientation_bitwise(lib):
    """One sample at the keypoint's own pixel (r2 = 0, weight exactly 1) for every fp32 angle within +-64 ulps of
    each bin boundary, near 0 and at float32(2 pi), and 5000 random angles: the oracle's output is bitwise the
    restatement's, and the bin decoded from it is the restated bin."""
    ang = R.angles_near_bin_edges(64, 5000, seed=0)
    n = len(ang)
    kp, grad = R.pack(np.zeros((n, 2)), R.sigma_for_orient_radius(1), (np.arange(n), 0, 0, 3.0, ang), 4)
    got = orc_orientations(lib, kp, grad)
    want, margin, _ = R.orientations(kp, grad, grad.shape[2], grad.shape[1], 1.0)
    assert np.array_equal(got.view(np.int32), want.view(np.int32)), int((got != want).any(axis=1).sum())
    assert np.isinf(margin).sum() == 0 and (margin > 0.01).all()
    dec = np.rint(got[:, 0].astype(np.float64) * 36 / R.TWO_PI - 0.5).astype(np.int64) % 36
    assert np.array_equal(dec, R.orient_bin(ang))
    assert R.orient_bin(np.float32(R.TWO_PI)) == 0 and np.float64(np.float32(R.TWO_PI)) > R.TWO_PI
    # the one-hot histogram path gives the same numbers
    onehot = np.zeros((n, R.NBINS), np.float32)
    onehot[np.arange(n), R.orient_bin(ang)] = 3.0
    assert np.array_equal(R.orient_from_hist(onehot)[0].view(np.int32), want.view(np.int32))


@pytest.mark.parametrize("W", [1, 2, 5, 10, 13])
def test_orientation_window_membership(lib, W):
    """One sample at every offset in [-11, 11]^2, keypoints on a 1/64 sub-pixel grid, inside the map and against
    every border and corner: the oracle's orientation is valid exactly when the restatement puts the sample in the
    clipped window (W = 13 is clamped to 10)."""
    s = R.sigma_for_orient_radius(W)
    offs = np.array([(a, b) for b in range(-11, 12) for a in range(-11, 12)])
    rng = np.random.default_rng(W)
    frac = np.repeat(rng.integers(0, 64, (4, 2)) / 64, len(offs), axis=0)
    frac[: len(offs)] = 0
    o = np.tile(offs, (4, 1))
    n = len(o)
    kp, grad = R.pack(frac, s, (np.arange(n), o[:, 0], o[:, 1], 1.0, 1.0), 26)
    x, y, _, xi, yi, _ = R.kp_geom(kp, 1.0)
    inside = R.in_orient_window(R.orient_r2(x, y, (xi + o[:, 0]).astype(np.float32), (yi + o[:, 1]).astype(np.float32)),
                                min(W, 10)) & (np.abs(o) <= min(W, 10)).all(axis=1)
    got = orc_orientations(lib, kp, grad)
    assert np.array_equal(got[:, 0] >= 0, inside)
    assert np.array_equal(R.orientations(kp, grad, grad.shape[2], grad.shape[1], 1.0)[0][:, 0] >= 0, inside)
    for frac_b in (0.0, 0.75):
        for kp, grad in R.pack_border(s, frac_b, offs):
            want = R.orientations(kp, grad, 50, 50, 1.0)[0]
            got = orc_orientations(lib, kp, grad)
            assert np.array_equal(got >= 0, want >= 0) and (ang_diff(got, want) <= FIT_ULPS).all()


def dense_case(seed, n=3000, ow=160, oh=120, smin=0.1):
    """Random dense gradient buffer (level 1 with a dominant direction, so that its histograms have clear peaks) and
    keypoints on a 1/64 grid anywhere in the octave, octave sigma smin .. 3 (0.1: every window radius)."""
    rng = np.random.default_rng(seed)
    grad = np.zeros((3, oh, ow, 2), np.float32)
    grad[..., 0] = rng.uniform(0, 10, (3, oh, ow))
    a = rng.random((3, oh, ow)) * R.TWO_PI
    a[1] = rng.vonmises(1.0, 2.0, (oh, ow)) % R.TWO_PI
    grad[..., 1] = np.minimum(a.astype(np.float32), np.float32(R.TWO_PI))
    kp = np.zeros((n, 4), np.float32)
    kp[:, 0] = rng.integers(0, (ow - 1) * 64, n) / 64
    kp[:, 1] = rng.integers(0, (oh - 1) * 64, n) / 64
    kp[:, 2] = rng.uniform(smin, 3.0, n)
    kp[:, 3] = rng.integers(0, 3, n)
    return kp, grad


def assert_orientations_within(got, want, margin, sens, eps, what):
    """Peak count and validity equal wherever the margin exceeds eps; angles within sens * eps + FIT_ULPS.
    Returns the number of keypoints decided by their margin."""
    dec = margin > eps
    assert np.array_equal(got[dec] >= 0, want[dec] >= 0), (what, np.nonzero(((got >= 0) != (want >= 0)).any(1) & dec)[0][:10])
    both = dec[:, None] & (got >= 0) & (want >= 0)
    d = ang_diff(got, want)
    bad = both & (d > sens * eps + FIT_ULPS)
    assert not bad.any(), (what, d[bad][:10], sens[bad][:10])
    return int((~dec).sum())


@pytest.mark.parametrize("seed", [11, 12])
def test_dense_orientations(lib, seed):
    kp, grad = dense_case(seed)
    got = orc_orientations(lib, kp, grad)
    want, margin, sens = R.orientations(kp, grad, grad.shape[2], grad.shape[1], 1.0)
    undecided = assert_orientations_within(got, want, margin, sens, ORACLE_EPS, "oracle")
    assert undecided < 0.05 * len(kp) and (want[:, 1] >= 0).sum() > 100


def test_impulse_descriptors(lib):
    """One sample at every offset of windows of 1, 2, 3 and 4 diagonal chunks, sub-pixel positions, random angle,
    th0 random or -1: every entry within 2^-20 * win * mod of the restatement, and exactly 0 where the sample is
    off the diagonal chunks, outside the window or outside the grid."""
    rng = np.random.default_rng(1)
    for W in (5, 12, 20, 28):
        offs = np.array([(a, b) for b in range(-W, W + 1) for a in range(-W, W + 1)])
        n = len(offs)
        kp, grad = R.pack(rng.integers(0, 64, (n, 2)) / 64, R.sigma_for_desc_radius(W),
                          (np.arange(n), offs[:, 0], offs[:, 1], rng.uniform(0.5, 20, n),
                           rng.random(n).astype(np.float32) * np.float32(R.TWO_PI)), 2 * W + 4, cols=64)
        th0 = rng.random(n).astype(np.float32) * np.float32(R.TWO_PI)
        th0[::7] = -1
        ori = np.stack([th0, -np.ones(n, np.float32)], 1)
        got, x, y = orc_descriptors(lib, kp, ori, grad)
        want, wm, valid = R.descriptors(kp, ori, grad, grad.shape[2], grad.shape[1], 3, 1.0)
        assert valid.all() and np.array_equal(x, kp[:, 0]) and np.array_equal(y, kp[:, 1])
        assert (np.abs(got - want) <= ORACLE_DESC * wm[:, None]).all(), W
        assert (got[wm == 0] == 0).all() and 0.1 < (wm > 0).mean() < 0.5


@pytest.mark.parametrize("seed", [11, 12])
def test_dense_descriptors(lib, seed):
    """Dense windows with the first orientation given (th0 = -1 for a fifth), num_dogs = 2 so that level-2
    keypoints fail the :49 check: every entry within 2^-20 * wm."""
    kp, grad = dense_case(seed, n=1500)
    rng = np.random.default_rng(seed)
    ori = np.stack([rng.random(len(kp)).astype(np.float32) * np.float32(R.TWO_PI), -np.ones(len(kp), np.float32)], 1)
    ori[::5, 0] = -1
    got, _, _ = orc_descriptors(lib, kp, ori, grad, num_dogs=2)
    want, wm, valid = R.descriptors(kp, ori, grad, grad.shape[2], grad.shape[1], 2, 1.0)
    assert np.array_equal(valid, kp[:, 3] < 2)
    assert (np.abs(got - want) <= ORACLE_DESC * wm[:, None]).all()
    assert (got[~valid] == 0).all() and (wm[valid] > 0).all()
