"""GPU suite: orient_kernel and describe_fast_kernel (niftymatch_b200/csrc/nm_orient_desc.cu) rule by rule against
the restatement of tests/orient_desc_ref.py (itself checked against the CPU oracle in tests/test_orient_desc_ref.py).

The compat entries nm_orientations_f32 / nm_descriptors_f32 run the same two kernels on any keypoint list and
gradient buffer, so each rule is driven with built inputs.  Most use impulse windows: every keypoint owns a cell of
a large gradient buffer and exactly one non-zero sample (or a few, where a rule needs them), and cells are far
enough apart that no window reaches another keypoint's samples.  A single sample at the keypoint's own pixel has
r2 = 0 and weight exactly 1, so its orientation is a fixed float function of its bin and is compared bitwise.
The last test runs the batched kernels (padded pitch, per-frame level offsets above 2^31 bytes, octave index from
the keypoint's meta word) on the benchmark's batch.

Bounds.
  * Histograms: the kernel sums a bin in lane-private fp32 partial sums (at most 14 samples per lane) and then over
    32 lanes, weights through ex2.approx (2 ulp, plus 2 x log2-argument rounding: 13 ulp for sigma >= 0.7); the
    restatement sums in float64 and rounds once; both smooth in the same 18 fp32 operations per bin.  The smoothed
    histograms therefore differ by a relative perturbation below (46 + 1 + 13 + 1 + 36) * 2^-24 < 2^-17 =
    KERNEL_EPS.  Peak decisions must agree wherever the restatement's margin exceeds it; angles may move by
    sens * KERNEL_EPS plus FIT_ULPS (1e-6 rad, the fp32 roundings of the fit).
  * Descriptors: per sample, the kernel's fp32 rotation (folded with 1 / SBP), bin arithmetic and ex2.approx window
    are within about 2^-19 of float64 relative to win * mod (the trilinear weights have slope <= 1 in nx, ny and nt,
    each within ~1e-6 of float64; the window's slope is nx / 4 <= 0.7); an entry is then summed in fp32 over at most
    64 samples per private copy and 16 copies (80 * 2^-24 = 2^-17.7 of the sum of its positive terms).  Every entry
    is held to 2^-16 * wm, wm the sum of win * mod of the samples that reach the grid; for an impulse that is the
    sample's own win * mod.  An impulse that reaches no cell must give exactly 0."""
import ctypes as C
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from niftymatch_b200 import synth  # noqa: E402
from tests import orient_desc_ref as R  # noqa: E402
from tests._util import ang_diff, orc_descriptors, orc_orientations  # noqa: E402
from tests.test_gpu_parity import DESC_REL_TOL, ORIENT_TOL  # noqa: E402
from tests.test_orient_desc_ref import ORACLE_EPS, dense_case  # noqa: E402

KERNEL_EPS = 2.0 ** -17
KERNEL_DESC = 2.0 ** -16
FIT_ULPS = 1e-6
TWO_PI_F = np.float32(R.TWO_PI)


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a, np.float32)).cuda()


def gpu_orient(nm, kp, grad, xper=1.0):
    out = nm.sift.orientations(_cu(kp), _cu(grad), grad.shape[2], grad.shape[1], xper)
    return out.cpu().numpy()


def gpu_desc(nm, kp, ori, grad, num_dogs=3, xper=1.0, sentinel=0.0):
    """nm_descriptors_f32 with the outputs filled with `sentinel` beforehand."""
    n = len(kp)
    desc = torch.full((n, 128), sentinel, dtype=torch.float32, device="cuda")
    x = torch.full((n,), sentinel, dtype=torch.float32, device="cuda")
    y = torch.full((n,), sentinel, dtype=torch.float32, device="cuda")
    k, o, g = _cu(kp), _cu(ori), _cu(grad)
    rc = nm._lib.load().nm_descriptors_f32(C.c_void_p(k.data_ptr()), C.c_void_p(o.data_ptr()), C.c_void_p(g.data_ptr()), n,
                                           grad.shape[2], grad.shape[1], num_dogs, C.c_float(xper),
                                           C.c_void_p(desc.data_ptr()), C.c_void_p(x.data_ptr()), C.c_void_p(y.data_ptr()),
                                           C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    return desc.cpu().numpy(), x.cpu().numpy(), y.cpu().numpy()


def decode_bin(theta):
    return np.rint(theta.astype(np.float64) * 36 / R.TWO_PI - 0.5).astype(np.int64) % 36


def bin_centre(b):
    return np.float32((np.asarray(b) + 0.5) * R.TWO_PI / 36)


def assert_orient_within(got, want, margin, sens, eps, tol=FIT_ULPS):
    """Validity and peak count equal wherever margin > eps; angles within sens * eps + tol.  Returns the worst
    angle gap, the worst gap over its bound and the keypoints decided by their margin (printed)."""
    dec = margin > eps
    flip = ((got >= 0) != (want >= 0)).any(axis=1)
    assert not (flip & dec).any(), np.nonzero(flip & dec)[0][:10]
    for i in np.nonzero(flip)[0]:
        print(f"  decided by margin: keypoint {i}: got {got[i]}, restated {want[i]}, margin {margin[i]:.3g}")
    both = dec[:, None] & (got >= 0) & (want >= 0)
    d = np.where(both, ang_diff(got, want), 0.0)
    bound = sens * eps + tol
    assert (d <= bound).all(), (d[d > bound][:10], sens[d > bound][:10])
    return d.max(initial=0.0), (d / bound).max(initial=0.0), int((~dec).sum())


# ------------------------------------------------------------------ 1. bin decision
def test_bin_decision_bitwise(nm):
    """Every fp32 angle within +-4096 ulps of each bin boundary k * 2 pi / 36 (the whole band of the double-division
    fallback, 1e-5 of the quotient), [0, 2e-6] sampled logarithmically, 0, float32(2 pi) and 10^6 random angles, as
    single samples at r2 = 0: the orientation is bitwise the restatement's."""
    ang = R.angles_near_bin_edges(4096, 10 ** 6, seed=3)
    n = len(ang)
    kp, grad = R.pack(np.zeros((n, 2)), R.sigma_for_orient_radius(1), (np.arange(n), 0, 0, 3.0, ang), 2, cols=1024)
    got = gpu_orient(nm, kp, grad)
    onehot = np.zeros((n, R.NBINS), np.float32)
    onehot[np.arange(n), R.orient_bin(ang)] = 3.0
    want = np.concatenate([R.orient_from_hist(onehot[i: i + 2 ** 17])[0] for i in range(0, n, 2 ** 17)])
    bad = (got.view(np.int32) != want.view(np.int32)).any(axis=1)
    assert not bad.any(), (int(bad.sum()), ang[bad][:8], got[bad][:4], want[bad][:4])
    assert np.array_equal(decode_bin(got[:, 0]), R.orient_bin(ang))
    print(f"\nbin decision: {n} angles bitwise")


# ------------------------------------------------------------------ 2. orientation window
RADII = list(range(1, 11)) + [13]


def test_orientation_window(nm):
    """One sample at every offset in [-11, 11]^2, for window radii 1..10 and one above the clamp, with the keypoint
    on a pixel, at three random 1/64 positions and at two positions that put the offset (W, 0) or (0, W) in
    r2 in (W^2 + 0.5, W^2 + 0.6); then keypoints against each border and corner.  The orientation is valid exactly
    when the restatement puts the sample in the clipped window, and then within FIT_ULPS of it."""
    offs = np.array([(a, b) for b in range(-11, 12) for a in range(-11, 12)])
    rng = np.random.default_rng(7)
    frac, sig = [], []
    for W in RADII:
        w = min(W, 10)
        t = np.float32(1 - 0.55 / (2 * w))
        for f in [(0, 0)] + [tuple(v) for v in rng.integers(0, 64, (3, 2)) / 64] + [(t, 0), (0, t)]:
            frac.append(np.tile(np.float32(f), (len(offs), 1)))
            sig.append(np.full(len(offs), R.sigma_for_orient_radius(W), np.float32))
    frac, sig = np.concatenate(frac), np.concatenate(sig)
    o = np.tile(offs, (len(frac) // len(offs), 1))
    n = len(o)
    kp, grad = R.pack(frac, sig, (np.arange(n), o[:, 0], o[:, 1], 1.0, 1.0), 26)
    x, y, s, xi, yi, _ = R.kp_geom(kp, 1.0)
    W = R.orient_radius(s)[1]
    r2 = R.orient_r2(x, y, (xi + o[:, 0]).astype(np.float32), (yi + o[:, 1]).astype(np.float32))
    inside = R.in_orient_window(r2, W) & (np.abs(o) <= W[:, None]).all(axis=1)
    band = inside & (r2 > W ** 2 + 0.5)
    assert band.sum() >= 2 * len(RADII), band.sum()
    got = gpu_orient(nm, kp, grad)
    assert np.array_equal(got[:, 0] >= 0, inside), np.nonzero((got[:, 0] >= 0) != inside)[0][:10]
    want = R.orientations(kp, grad, grad.shape[2], grad.shape[1], 1.0)[0]
    assert np.array_equal(got >= 0, want >= 0) and (ang_diff(got, want) <= FIT_ULPS).all()
    calls = 0
    for Wb in (1, 4, 10, 13):
        for fb in (0.0, 0.75):
            for kp, grad in R.pack_border(R.sigma_for_orient_radius(Wb), fb, offs):
                want = R.orientations(kp, grad, 50, 50, 1.0)[0]
                got = gpu_orient(nm, kp, grad)
                assert np.array_equal(got >= 0, want >= 0), (Wb, fb, got[:, 0], want[:, 0])
                assert (ang_diff(got, want) <= FIT_ULPS).all()
                calls += 1
    print(f"\norientation window: {n} interior impulses ({int(band.sum())} in the r2 band above W^2 + 0.5), "
          f"{calls} border maps")


# ------------------------------------------------------------------ 3. peak rules
def _peaks(nm, samples, n, s=R.sigma_for_orient_radius(3)):
    """Keypoints on a pixel with the given samples: kernel and restatement results."""
    kp, grad = R.pack(np.zeros((n, 2)), s, samples, 16)
    return gpu_orient(nm, kp, grad), R.orientations(kp, grad, grad.shape[2], grad.shape[1], 1.0)


def test_empty_window_and_negative_level(nm):
    """An all-zero window gives (-1, -1); so does kp.w < 0 whatever its window holds."""
    kp, grad = R.pack(np.zeros((6, 2)), 1.0, (np.array([3, 4, 5]), 0, 0, 2.0, 1.0), 16)
    kp[3:, 3] = -1
    got = gpu_orient(nm, kp, grad)
    assert (got == -1).all()


def test_three_peaks_first_two_in_bin_order(nm):
    """Three equal samples at r2 = 1 in bins at least 10 apart (circularly), including bins 32-35 and triples that
    wrap past bin 0: the orientations are the two lowest bins, ascending, within FIT_ULPS of the restatement."""
    tri = np.array([(a, b, c) for a in range(36) for b in range(a + 10, 36) for c in range(b + 10, 36) if a + 36 - c >= 10])
    assert (tri >= 32).any(axis=1).sum() > 0
    rng = np.random.default_rng(9)
    tri = np.array([rng.permutation(t) for t in tri])          # the sample order in the window is not the bin order
    n = len(tri)
    k = np.repeat(np.arange(n), 3)
    ox = np.tile([1, 0, -1], n)
    oy = np.tile([0, 1, 0], n)
    got, (want, margin, sens) = _peaks(nm, (k, ox, oy, 2.0, bin_centre(tri.reshape(-1))), n)
    lo = np.sort(tri, axis=1)[:, :2]
    assert np.array_equal(decode_bin(got[:, 0]), lo[:, 0]) and np.array_equal(decode_bin(got[:, 1]), lo[:, 1])
    assert_orient_within(got, want, margin, sens, KERNEL_EPS)
    print(f"\nthree peaks: {n} triples, {int((tri >= 32).any(axis=1).sum())} with a bin in 32-35")


def test_second_peak_threshold_sweep(nm):
    """Two samples at equal r2 (same ex2.approx weight) in bins 17 apart, the second's magnitude swept through 0.8 of
    the first (every fp32 ratio within 64 ulps of 0.8 and a grid from 0.79 to 0.81), in both bin orders: the second
    orientation switches on exactly once, within 1e-5 of 0.8, and agrees with the restatement off its margin."""
    r = np.concatenate([np.arange(np.float32(0.8).view(np.int32) - 64, np.float32(0.8).view(np.int32) + 65,
                                  dtype=np.int32).view(np.float32), np.linspace(0.79, 0.81, 2001, dtype=np.float32)])
    r = np.unique(r)
    for big, small in ((4, 21), (30, 13)):
        n = len(r)
        k = np.repeat(np.arange(n), 2)
        mod = np.stack([np.ones(n, np.float32), r], 1).reshape(-1)
        ang = np.tile(bin_centre([big, small]), n)
        got, (want, margin, sens) = _peaks(nm, (k, np.tile([1, -1], n), 0, mod, ang), n)
        on = (got >= 0).sum(axis=1) == 2
        assert (got[:, 0] >= 0).all()
        sw = np.nonzero(np.diff(on.astype(int)))[0]
        assert len(sw) == 1 and not on[0] and on[-1], sw
        assert abs(float(r[sw[0] + 1]) - 0.8) <= 1e-5 and abs(float(r[sw[0]]) - 0.8) <= 1e-5, r[sw[0]: sw[0] + 2]
        assert (decode_bin(got[:, 0]) == np.where(on, min(big, small), big)).all()
        assert_orient_within(got, want, margin, sens, KERNEL_EPS)


def test_adjacent_bin_parabolic_fit(nm):
    """Two samples at equal r2 in adjacent bins b, b + 1 (mod 36) with magnitude ratios 0.3 .. 1: the fitted angle
    is within FIT_ULPS + sens * KERNEL_EPS of the restatement's."""
    b = np.repeat(np.arange(36), 8)
    ratio = np.tile(np.linspace(0.3, 1.0, 8, dtype=np.float32), 36)
    n = len(b)
    k = np.repeat(np.arange(n), 2)
    mod = np.stack([np.full(n, 1.5, np.float32), 1.5 * ratio], 1).reshape(-1)
    ang = np.stack([bin_centre(b), bin_centre((b + 1) % 36)], 1).reshape(-1)
    got, (want, margin, sens) = _peaks(nm, (k, np.tile([0, 0], n), np.tile([1, -1], n), mod, ang), n)
    assert (got[:, 0] >= 0).all()
    worst = assert_orient_within(got, want, margin, sens, KERNEL_EPS)
    print(f"\nparabolic fit: {n} pairs, worst gap {worst[0]:.3g} rad")


def test_positive_exponent_window(nm):
    """Two samples of equal magnitude in bins 17 apart, one at the keypoint (weight 1) and one at r2 = W^2, whose
    weight exp(+W^2 / 2 sigma_w^2) exceeds 1 / 0.8: only the far sample's peak survives."""
    rows = []
    for W in (2, 3, 5, 8, 10):
        for near_bin, far_bin in ((5, 22), (22, 5)):
            rows.append((W, near_bin, far_bin))
    rows = np.array(rows)
    n = len(rows)
    k = np.repeat(np.arange(n), 2)
    ox = np.stack([np.zeros(n, int), rows[:, 0]], 1).reshape(-1)
    ang = np.stack([bin_centre(rows[:, 1]), bin_centre(rows[:, 2])], 1).reshape(-1)
    s = np.array([R.sigma_for_orient_radius(W) for W in rows[:, 0]], np.float32)
    sw = R.orient_radius(s)[0].astype(np.float64)
    assert (np.exp(rows[:, 0] ** 2 / (2 * sw ** 2)) > 1 / 0.8).all()
    kp, grad = R.pack(np.zeros((n, 2)), s, (k, ox, 0, 2.0, ang), 24)
    got = gpu_orient(nm, kp, grad)
    assert np.array_equal(decode_bin(got[:, 0]), rows[:, 2]) and (got[:, 1] == -1).all(), got


# ------------------------------------------------------------------ 4. descriptor impulses
TH0 = np.concatenate([np.float32([0, np.pi / 2, np.pi, 3 * np.pi / 2, -1]), [np.nextafter(TWO_PI_F, np.float32(0))],
                      np.random.default_rng(21).random(16).astype(np.float32) * TWO_PI_F]).astype(np.float32)
DESC_RADII = (5, 12, 20, 28)            # 1, 2, 3 and 4 diagonal chunks


def _desc_check(nm, kp, ori, grad, num_dogs=3):
    got, x, y = gpu_desc(nm, kp, ori, grad, num_dogs)
    want, wm, valid = R.descriptors(kp, ori, grad, grad.shape[2], grad.shape[1], num_dogs, 1.0)
    assert valid.all() and np.array_equal(x, kp[:, 0]) and np.array_equal(y, kp[:, 1])
    gap = np.abs(got - want)
    assert (got[wm == 0] == 0).all(), np.nonzero((got[wm == 0] != 0).any(axis=1))[0][:10]
    bad = (gap > KERNEL_DESC * wm[:, None]).any(axis=1)
    assert not bad.any(), (np.nonzero(bad)[0][:10], (gap.max(axis=1) / wm)[bad][:10])
    nz = wm > 0
    return (gap.max(axis=1)[nz] / wm[nz]).max(initial=0.0), int(nz.sum()), int((~nz).sum())


@pytest.mark.parametrize("W", DESC_RADII)
def test_descriptor_impulses(nm, W):
    """One sample at every offset of the window, the keypoint on a pixel or at a random 1/64 position, th0 cycling
    through 0, pi/2, pi, 3 pi/2, -1, the float below 2 pi and 16 random angles, random sample angle and magnitude:
    every entry within 2^-16 * win * mod of the restatement, exactly 0 when the sample reaches no cell (off the
    diagonal chunks, outside the window or outside the 4 x 4 grid), x and y the keypoint's."""
    rng = np.random.default_rng(W)
    offs = np.array([(a, b) for b in range(-W - 2, W + 3) for a in range(-W - 2, W + 3)])
    offs = np.tile(offs, (2, 1))
    n = len(offs)
    frac = rng.integers(0, 64, (n, 2)) / 64
    frac[: n // 2] = 0
    kp, grad = R.pack(frac, R.sigma_for_desc_radius(W), (np.arange(n), offs[:, 0], offs[:, 1], rng.uniform(0.5, 20, n),
                                                        rng.random(n).astype(np.float32) * TWO_PI_F), 2 * W + 8, cols=64)
    ori = np.stack([TH0[np.arange(n) % len(TH0)], np.full(n, -1, np.float32)], 1)
    worst, reach, zero = _desc_check(nm, kp, ori, grad)
    print(f"\ndescriptor impulses W = {W}: {n}, {reach} reach the grid, worst entry gap / (win * mod) = {worst:.3g} "
          f"(2^{math.log2(worst) if worst else float('-inf'):.2f})")


def test_descriptor_impulses_clipped_windows(nm):
    """Keypoints against each border and corner (window radius 12), and a 20 x 20 octave smaller than a radius-28
    window: impulses at every offset inside the octave, every entry within bounds, exact zeros elsewhere."""
    rng = np.random.default_rng(4)
    offs = np.array([(a, b) for b in range(-13, 14) for a in range(-13, 14)])
    worst = 0.0
    for fb in (0.0, 0.5):
        for kp, grad in R.pack_border(R.sigma_for_desc_radius(12), fb, offs, size=56):
            m = grad[..., 0] > 0
            grad[..., 0][m] = rng.uniform(0.5, 20, m.sum())
            grad[..., 1][m] = rng.random(m.sum()) * TWO_PI_F
            ori = np.stack([TH0[rng.integers(0, len(TH0), 24)], np.full(24, -1, np.float32)], 1)
            worst = max(worst, _desc_check(nm, kp, ori, grad)[0])
    size = 20
    px = np.array([(a, b) for b in range(size) for a in range(size)])
    kp = np.tile(np.float32([[9.25, 10.5, R.sigma_for_desc_radius(28), 0]]), (3, 1))
    kp[:, 3] = [0, 1, 2]
    for r in range(-(-len(px) // 3)):
        grad = np.zeros((3, size, size, 2), np.float32)
        for lev in range(3):
            if 3 * r + lev < len(px):
                grad[lev, px[3 * r + lev, 1], px[3 * r + lev, 0]] = (rng.uniform(0.5, 20), rng.random() * TWO_PI_F)
        ori = np.stack([TH0[rng.integers(0, len(TH0), 3)], np.full(3, -1, np.float32)], 1)
        worst = max(worst, _desc_check(nm, kp, ori, grad)[0])
    print(f"\nclipped descriptor windows: worst entry gap / (win * mod) = {worst:.3g}")


def test_descriptor_slots_failing_the_range_check_keep_their_contents(nm):
    """Keypoints whose pixel is outside the octave (left, right, above, below) and level-2 keypoints with
    num_dogs = 2 leave their descriptor, x and y slots as they were; the others are computed."""
    kp, grad = dense_case(5, n=60, ow=64, oh=48, smin=0.7)
    kp[:, 3] = np.arange(60) % 3
    kp[0:4, :2] = [(-3.0, 10.0), (66.5, 10.0), (10.0, -2.0), (10.0, 48.6)]
    kp[0:4, 3] = 0
    ori = np.stack([np.random.default_rng(5).random(60).astype(np.float32) * TWO_PI_F, np.full(60, -1, np.float32)], 1)
    got, x, y = gpu_desc(nm, kp, ori, grad, num_dogs=2, sentinel=-7.0)
    want, wm, valid = R.descriptors(kp, ori, grad, 64, 48, 2, 1.0)
    assert not valid[:4].any() and np.array_equal(valid[4:], kp[4:, 3] < 2)
    assert (got[~valid] == -7.0).all() and (x[~valid] == -7.0).all() and (y[~valid] == -7.0).all()
    assert np.array_equal(x[valid], kp[valid, 0]) and np.array_equal(y[valid], kp[valid, 1])
    assert (np.abs(got[valid] - want[valid]) <= KERNEL_DESC * wm[valid, None]).all()


# ------------------------------------------------------------------ 5. dense random windows
@pytest.mark.parametrize("seed", [31, 32])
def test_dense_windows(nm, oracle, seed):
    """Dense random gradient buffers, keypoints anywhere in the octave (sigma 0.7 .. 3), against the restatement
    (margins, sensitivity, 2^-16 * wm) and against the oracle (ORIENT_TOL and DESC_REL_TOL, decisions off the
    margins of both)."""
    kp, grad = dense_case(seed, n=4000, smin=0.7)
    oh, ow = grad.shape[1:3]
    got = gpu_orient(nm, kp, grad)
    want, margin, sens = R.orientations(kp, grad, ow, oh, 1.0)
    worst, ratio, undecided = assert_orient_within(got, want, margin, sens, KERNEL_EPS)
    orc = orc_orientations(oracle.lib, kp, grad)
    assert_orient_within(got, orc, margin, sens, KERNEL_EPS + ORACLE_EPS, ORIENT_TOL)
    ori = got.copy()
    ori[::7, 0] = -1
    d, x, y = gpu_desc(nm, kp, ori, grad)
    dw, wm, valid = R.descriptors(kp, ori, grad, ow, oh, 3, 1.0)
    assert valid.all() and (wm > 0).all()
    gap = np.abs(d - dw).max(axis=1) / wm
    assert (gap <= KERNEL_DESC).all(), gap.max()
    do = orc_descriptors(oracle.lib, kp, ori, grad)[0]
    rel = np.linalg.norm(d - do, axis=1) / np.maximum(np.linalg.norm(do, axis=1), 1e-20)
    assert rel.max() <= DESC_REL_TOL, rel.max()
    print(f"\ndense windows: orientation worst gap {worst:.3g} rad ({ratio:.3g} of its bound), {undecided} of {len(kp)} "
          f"decided by margin; descriptor worst entry gap / wm = {gap.max():.3g} (2^{math.log2(gap.max()):.2f}), "
          f"vs oracle rel L2 {rel.max():.3g}")


# ------------------------------------------------------------------ 6. the batched path at the benchmark shape
BENCH_N, BENCH_CAP = 64, 16384


def check_frame(kpts, ori, desc, seg, grads, num_dogs, eps):
    """One frame's keypoints (segment order), orientations and descriptors against the restatement on the frame's
    gradient maps grads[o] (3, oh, ow, 2): orientations within ORIENT_TOL + sens * eps off the margin, every
    descriptor entry within 2^-16 * wm.  Returns the measured gaps."""
    nk = len(kpts)
    want, margin, sens = np.zeros_like(ori), np.zeros(nk), np.zeros((nk, 2))
    dwant, wm = np.zeros((nk, 128)), np.zeros(nk)
    start = 0
    for o, grad in enumerate(grads):
        oh, ow = grad.shape[1:3]
        for l in range(3):
            sl = slice(start, start + int(seg[3 * o + l]))
            start = sl.stop
            if sl.stop == sl.start:
                continue
            assert (kpts[sl, 3] == l).all()
            want[sl], margin[sl], sens[sl] = R.orientations(kpts[sl], grad, ow, oh, 2.0 ** o)
            dwant[sl], wm[sl], valid = R.descriptors(kpts[sl], ori[sl], grad, ow, oh, num_dogs, 2.0 ** o)
            assert valid.all()
    assert start == nk
    worst, ratio, undecided = assert_orient_within(ori, want, margin, sens, eps, ORIENT_TOL)
    gap = np.abs(desc - dwant[: len(desc)]).max(axis=1) / np.maximum(wm[: len(desc)], 1e-30)
    assert (desc[wm[: len(desc)] == 0] == 0).all()
    assert (gap <= KERNEL_DESC).all(), (np.nonzero(gap > KERNEL_DESC)[0][:10], gap.max())
    return worst, ratio, undecided, gap.max()


def test_benchmark_batch_every_keypoint(nm, oracle):
    """The benchmark's 64 x 1080p batch with dense gradient maps.  For frames 0, 31 and 63, keypoints are split by
    segment (octave o, level l; xper = 2^o) and checked against the restatement on the frame's own gradient maps:
    every orientation within ORIENT_TOL + sens * KERNEL_EPS (validity and peak count may differ only below the
    margin, and each such keypoint is printed), and every descriptor, computed from the product's orientations,
    within 2^-16 * wm per entry -- no keypoint exempt.  The oracle, given the product's orientations, agrees to
    DESC_REL_TOL."""
    frames = np.stack([synth.scene(1920, 1080, synth.SEED_BASE + g) for g in range(BENCH_N)])
    P = nm.SiftParams(1920, 1080)
    sb = nm.SiftBatch(P, BENCH_N, BENCH_CAP)
    sb.set_dense_gradients(True)
    sb.run(_cu(frames))
    torch.cuda.synchronize()
    r = sb.results()
    stats = []
    for f in (0, BENCH_N // 2 - 1, BENCH_N - 1):
        seg = r["seg_counts"][f].cpu().numpy()
        nk = int(seg.sum())
        c = int(r["counts"][f].item())
        assert nk <= BENCH_CAP and c == nk and c > 5000, (nk, c)
        kpts = r["kpts"][f, :nk].cpu().numpy()
        ori = r["orient"][f, :nk].cpu().numpy()
        desc = r["desc"][f, :c].cpu().numpy()
        assert np.array_equal(r["x"][f, :c].cpu().numpy(), kpts[:, 0]) and np.array_equal(r["y"][f, :c].cpu().numpy(), kpts[:, 1])
        grads = [np.stack([sb.grad(f, o, l).cpu().numpy() for l in range(3)]) for o in range(sb.n_oct)]
        worst, ratio, undecided, gap = check_frame(kpts, ori, desc, seg, grads, P._num_dog_levels, KERNEL_EPS)
        co = oracle.sift_frame(frames[f], capacity=BENCH_CAP, orient_mode=2, orient_in=ori, want_levels=False)
        assert co["n"] == c and np.array_equal(co["kpts"], kpts)
        rel = np.linalg.norm(desc - co["desc"], axis=1) / np.maximum(np.linalg.norm(co["desc"], axis=1), 1e-20)
        assert rel.max() <= DESC_REL_TOL, rel.max()
        stats.append((f, nk, worst, ratio, undecided, gap, rel.max()))
    sb.close()
    torch.cuda.empty_cache()
    for f, nk, worst, ratio, undecided, g, rel in stats:
        print(f"\nbatch frame {f}: {nk} keypoints; orientation worst gap {worst:.3g} rad ({ratio:.3g} of its bound), "
              f"{undecided} decided by margin; descriptor worst entry gap / wm {g:.3g} (2^{math.log2(g):.2f}), "
              f"vs oracle rel L2 {rel:.3g}")
