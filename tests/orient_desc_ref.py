"""Restatement of the reference's orientation (gpu/kernels/orientation.cu:11-129) and descriptor
(gpu/kernels/descriptor.cu:32-145) semantics in numpy, vectorised over keypoints.  Test helper: the CPU oracle
(oracle/nm_oracle.c) and the CUDA kernels (niftymatch_b200/csrc/nm_orient_desc.cu) are both checked against it.

Orientation.  Every discrete decision is reproduced with the IEEE fp32 / fp64 operations of the reference: keypoint
geometry and the window radius W, the window test (double)r2 < W*W + 0.6 with r2 = fmaf(dx, dx, dy*dy), the bin
floor((float)((double)(36 v) / 2 pi)) mod 36, the six 3-tap smoothing passes, the maximum, the 0.8 threshold and the
parabolic fit of the first two peaks.  Only the sample weights exp(+r2 / 2 sigma_w^2) and their sum per bin are
computed in float64 (rounded to fp32 once, before the smoothing): kernels sum in other orders and with other exp
approximations, so a histogram is reproduced up to a small relative perturbation.  For every keypoint the function
therefore also returns
  * margin: the smallest uniform relative perturbation of the smoothed histogram that can flip one of the peak
    decisions (h0 > thr, h0 > hm, h0 > hp) up to the bin that decides the output;
  * sens: for each returned angle, the largest change of the angle (rad) per unit relative perturbation of the three
    bins of its parabolic fit (first-order, from the fit's derivative).
A window with exactly one non-zero sample at r2 = 0 has weight 1 everywhere, so its result is exact.

Descriptor.  Float64 throughout, with the reference's semantics: first orientation only (th0 = -1 is taken
literally), the window clipped to the octave, only the diagonal 16 x 16 chunks of the window visited, trilinear
spread into a 4 x 4 x 8 grid with the (bint + dbt) % 8 wrap, no normalisation.  The descriptor is continuous in
the sample position and angle, so float64 needs no exclusions.  Also returned per keypoint: wm, the sum of
win * mod over the visited samples whose rotated position is within 1e-4 of the grid's support (|nx|, |ny| < 2.5),
the scale of every per-entry error bound; a keypoint with wm = 0 has an all-zero descriptor in every
implementation."""
from __future__ import annotations

import numpy as np

F32 = np.float32
TWO_PI = 2 * np.pi                 # 2 * M_PI in double
NBINS = 36
ORIENT_WMAX = 10                   # the reference's 22 x 22 block clamps the orientation window


# ------------------------------------------------------------------ inputs
def pack(frac, s, samples, spacing, cols=256, levels=3):
    """Keypoints with sparse windows in one gradient buffer.  Keypoint k sits on level k % levels, in cell k // levels
    of a grid of spacing x spacing cells (cols per row), at its cell's centre pixel plus frac[k] (in [0, 1)^2).
    samples = (k, ox, oy, mod, ang) arrays: sample i is written at offset (ox, oy) from the nearest pixel of keypoint
    k[i].  A spacing above the window diameter plus the largest offset keeps every window clear of the other
    keypoints' samples.  Returns kp (n, 4) and grad (levels, oh, ow, 2), with xper = 1."""
    frac = np.asarray(frac, np.float32).reshape(-1, 2)
    n = len(frac)
    cell = np.arange(n) // levels
    rows = -(-int(cell.max() + 1) // cols)
    ncols = min(cols, int(cell.max()) + 1)
    ow, oh = ncols * spacing, rows * spacing
    kp = np.zeros((n, 4), np.float32)
    kp[:, 0] = (cell % cols) * spacing + spacing // 2 + frac[:, 0]
    kp[:, 1] = (cell // cols) * spacing + spacing // 2 + frac[:, 1]
    kp[:, 2] = s
    kp[:, 3] = np.arange(n) % levels
    _, _, _, xi, yi, lev = kp_geom(kp, 1.0)
    k, ox, oy, mod, ang = samples
    k = np.asarray(k, np.int64)
    grad = np.zeros((levels, oh, ow, 2), np.float32)
    grad[lev[k], yi[k] + np.asarray(oy, np.int64), xi[k] + np.asarray(ox, np.int64)] = np.stack(
        [np.broadcast_to(np.float32(mod), k.shape), np.broadcast_to(np.float32(ang), k.shape)], axis=-1)
    return kp, grad


def pack_border(s, frac, offsets, size=50):
    """Maps of size x size with 8 keypoints per level against the borders and corners: x and y each in {frac, the
    centre, size - 1 - frac} except the centre itself.  Round r gives keypoint j on level l the offset r * levels + l
    of those of `offsets` that stay inside the map (none once they run out).  Yields kp (24, 4), grad (3, size,
    size, 2); every sample has mod 1 and angle 1."""
    a, c, b = frac, size // 2, size - 1 - frac
    pos = np.array([(x, y) for y in (a, c, b) for x in (a, c, b) if (x, y) != (c, c)], np.float32)
    kp = np.zeros((24, 4), np.float32)
    kp[:, :2] = np.repeat(pos, 3, axis=0)
    kp[:, 2] = s
    kp[:, 3] = np.tile(np.arange(3), 8)
    _, _, _, xi, yi, _ = kp_geom(kp, 1.0)
    offsets = np.asarray(offsets, np.int64).reshape(-1, 2)
    own = [offsets[(xi[j] + offsets[:, 0] >= 0) & (xi[j] + offsets[:, 0] < size) &
                   (yi[j] + offsets[:, 1] >= 0) & (yi[j] + offsets[:, 1] < size)] for j in range(24)]
    for r in range(-(-max(len(o) for o in own) // 3)):
        grad = np.zeros((3, size, size, 2), np.float32)
        for j in range(24):
            i = 3 * r + j % 3
            if i < len(own[j]):
                grad[j % 3, yi[j] + own[j][i, 1], xi[j] + own[j][i, 0]] = (1.0, 1.0)
        yield kp, grad


def angles_near_bin_edges(ulps, n_random, seed):
    """Every fp32 angle within +-ulps of the bin boundaries k * 2 pi / 36, k = 1..36, 0 and float32(2 pi), 512
    angles in [0, 2e-6] spaced logarithmically (at k = 0 the band holds too many floats), and n_random uniform
    angles; all in [0, float32(2 pi)]."""
    two_pi = np.float32(TWO_PI)
    out = [np.float32([0.0, two_pi]), np.geomspace(1e-38, 2e-6, 512).astype(np.float32),
           np.random.default_rng(seed).random(n_random).astype(np.float32) * two_pi]
    for k in range(1, 37):
        b = np.float32(k * TWO_PI / 36).view(np.int32)
        out.append(np.arange(b - ulps, b + ulps + 1, dtype=np.int32).view(np.float32))
    a = np.concatenate(out)
    return a[(a >= 0) & (a <= two_pi)]


def sigma_for_orient_radius(W):
    """An octave sigma s whose orientation window radius floor(4.5 s) is W (W > 10: clamped to 10)."""
    return np.float32((W + 0.5) / 4.5)


def sigma_for_desc_radius(W):
    """An octave sigma s whose descriptor window radius floor(3 s * 5 / sqrt(2) + 0.5) is W."""
    return np.float32(W / (3 * 5 / np.sqrt(2.0)))


# ------------------------------------------------------------------ geometry (orientation.cu:19-30, descriptor.cu:41-65)
def kp_geom(kp, xper):
    """Octave coordinates (fp32), nearest pixel ((int)((double)x + 0.5)) and level of (n, 4) keypoints."""
    kp = np.asarray(kp, np.float32).reshape(-1, 4)
    xp = F32(xper)
    x, y, s = kp[:, 0] / xp, kp[:, 1] / xp, kp[:, 2] / xp
    xi = np.trunc(x.astype(np.float64) + 0.5).astype(np.int64)
    yi = np.trunc(y.astype(np.float64) + 0.5).astype(np.int64)
    return x, y, s, xi, yi, np.trunc(kp[:, 3]).astype(np.int64)


def orient_radius(s):
    """sigma_w = 1.5 s and W = min(max(floor(3 sigma_w), 1), 10)."""
    sigma_w = F32(1.5) * np.asarray(s, np.float32)
    W = np.maximum(np.floor(F32(3) * sigma_w).astype(np.int64), 1)
    return sigma_w, np.minimum(W, ORIENT_WMAX)


def fmaf(a, b, c):
    """Correctly rounded fp32 fma(a, b, c) of fp32 arrays.  a * b is exact in double; the double sum a * b + c is
    rounded once more, which can only go wrong when it lands exactly on the midpoint of two floats: the exact
    remainder of the sum (TwoSum) then decides."""
    p = np.asarray(a, np.float64) * np.asarray(b, np.float64)
    c = np.asarray(c, np.float64)
    s = p + c
    bb = s - p
    err = (p - (s - bb)) + (c - bb)
    r = s.astype(np.float32)
    lo = np.where(r.astype(np.float64) > s, np.nextafter(r, F32(-np.inf)), r)
    hi = np.nextafter(lo, F32(np.inf))
    tie = (err != 0) & (s == (lo.astype(np.float64) + hi.astype(np.float64)) / 2)
    return np.where(tie, np.where(err > 0, hi, lo), r).astype(np.float32)


def orient_r2(x, y, px, py):
    """r2 = fmaf(dx, dx, dy * dy) of a sample at octave pixel (px, py) from the keypoint at (x, y) (:52-54)."""
    dx = np.asarray(px, np.float32) - np.asarray(x, np.float32)
    dy = np.asarray(py, np.float32) - np.asarray(y, np.float32)
    return fmaf(dx, dx, dy * dy)


def in_orient_window(r2, W):
    """:55 (double)r2 < W * W + 0.6."""
    return np.asarray(r2, np.float32).astype(np.float64) < (np.asarray(W, np.int64) ** 2).astype(np.float64) + 0.6


def orient_bin(ang):
    """:57-58 floor((float)((double)(36 v) / 2 pi)) % 36 of fp32 angles in [0, float32(2 pi)]."""
    v36 = F32(36) * np.asarray(ang, np.float32)
    q = (v36.astype(np.float64) / TWO_PI).astype(np.float32)
    return np.floor(q).astype(np.int64) % NBINS


# ------------------------------------------------------------------ orientation
def orient_from_hist(hist):
    """Smoothing, threshold and peak fit (orientation.cu:71-128) of (n, 36) fp32 histograms.
    Returns theta (n, 2) fp32 (-1 where absent), margin (n,) and sens (n, 2) (see the module docstring)."""
    h = np.asarray(hist, np.float32).reshape(-1, NBINS)
    n = h.shape[0]
    for _ in range(6):
        h = ((np.roll(h, 1, axis=1) + h) + np.roll(h, -1, axis=1)) / F32(3)
    m = np.maximum(F32(0), h.max(axis=1))
    thr = (m.astype(np.float64) * 0.8).astype(np.float32)
    hm, hp = np.roll(h, 1, axis=1), np.roll(h, -1, axis=1)
    peak = (h > thr[:, None]) & (h > hm) & (h > hp)
    b = np.arange(NBINS, dtype=np.float32)[None, :]
    num = -0.5 * (hp - hm).astype(np.float64)
    dn = ((hp + hm) - F32(2) * h).astype(np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        di = (num / dn).astype(np.float32)
        th = (TWO_PI * ((b + di).astype(np.float64) + 0.5) / 36).astype(np.float32)
        h64, hm64, hp64 = h.astype(np.float64), hm.astype(np.float64), hp.astype(np.float64)
        sens = (TWO_PI / 36) * (np.abs(h64 - hm64) * hp64 + np.abs(hp64 - h64) * hm64 + np.abs(hp64 - hm64) * h64) / dn ** 2
        # relative perturbation that flips each decision: x > y fails once x (1 - e) <= y (1 + e)
        t64 = thr.astype(np.float64)[:, None]
        flip = np.minimum(np.minimum(np.abs(h64 - t64) / (h64 + t64), np.abs(h64 - hm64) / (h64 + hm64)),
                          np.abs(h64 - hp64) / (h64 + hp64))
    flip = np.where(np.isnan(flip), np.inf, flip)      # 0 > 0 between empty bins: exact in every implementation
    theta = np.full((n, 2), -1, np.float32)
    s_out = np.zeros((n, 2))
    rank = np.cumsum(peak, axis=1)                       # peaks found up to and including each bin
    for k in range(2):
        sel = peak & (rank == k + 1)
        has = sel.any(axis=1)
        idx = sel.argmax(axis=1)
        theta[has, k] = th[has, idx[has]]
        s_out[has, k] = sens[has, idx[has]]
    # the decisions up to the third peak fix the output (a change past it moves neither of the first two)
    last = np.where(rank[:, -1] >= 3, (rank >= 3).argmax(axis=1), NBINS - 1)
    upto = np.arange(NBINS)[None, :] <= last[:, None]
    margin = np.where(upto, flip, np.inf).min(axis=1)
    margin = np.where(m > 0, margin, np.inf)             # an all-zero histogram is decided exactly
    return theta, margin, s_out


def orient_hist(kp, grad, ow, oh, xper, block=4096):
    """(n, 36) fp32 histograms of the clipped windows (:32-58); grad is the (levels, oh, ow, 2) gradient buffer of
    the octave.  Keypoints with kp.w < 0 get an all-zero histogram."""
    x, y, s, xi, yi, lev = kp_geom(kp, xper)
    sigma_w, W = orient_radius(s)
    n = len(x)
    out = np.zeros((n, NBINS), np.float32)
    off = np.arange(-ORIENT_WMAX, ORIENT_WMAX + 1)
    for b0 in range(0, n, block):
        sl = slice(b0, min(n, b0 + block))
        cx, cy = off[None, None, :], off[None, :, None]
        Wb, xib, yib = W[sl, None, None], xi[sl, None, None], yi[sl, None, None]
        inside = ((cx >= np.maximum(-Wb, -xib)) & (cx <= np.minimum(Wb, ow - 1 - xib)) &
                  (cy >= np.maximum(-Wb, -yib)) & (cy <= np.minimum(Wb, oh - 1 - yib)))
        px, py = xib + cx, yib + cy
        r2 = orient_r2(x[sl, None, None], y[sl, None, None], px.astype(np.float32), py.astype(np.float32))
        use = inside & in_orient_window(r2, Wb) & (np.asarray(kp, np.float32)[sl, 3] >= 0)[:, None, None]
        k, iy, ix = np.nonzero(use)
        g = grad[lev[sl][k], py[k, iy, 0], px[k, 0, ix]]
        sw = sigma_w[sl][k].astype(np.float64)
        wgt = np.exp(r2[k, iy, ix].astype(np.float64) / (2 * sw * sw))
        acc = np.zeros((sl.stop - sl.start, NBINS))
        np.add.at(acc, (k, orient_bin(g[:, 1])), g[:, 0].astype(np.float64) * wgt)
        out[sl] = acc.astype(np.float32)
    return out


def orientations(kp, grad, ow, oh, xper):
    """theta (n, 2), margin (n,), sens (n, 2) of keypoints on one octave's gradient buffer."""
    return orient_from_hist(orient_hist(kp, grad, ow, oh, xper))


# ------------------------------------------------------------------ descriptor
def desc_window(s, xi, yi, ow, oh):
    """SBP (fp32), the clipped window [xmin, xmax] x [ymin, ymax] and the number of diagonal chunks (:54-65)."""
    SBP = ((F32(3) * np.asarray(s, np.float32)).astype(np.float64) + 1e-07).astype(np.float32)
    W = np.floor(np.sqrt(2.0) * SBP.astype(np.float64) * 5 / 2.0 + 0.5).astype(np.int64)
    xmin, xmax = np.maximum(-W, -xi), np.minimum(W, ow - 1 - xi)
    ymin, ymax = np.maximum(-W, -yi), np.minimum(W, oh - 1 - yi)
    chunks = np.ceil((np.maximum(xmax - xmin, ymax - ymin) + F32(1)) / F32(16)).astype(np.int64)
    return SBP, W, xmin, xmax, ymin, ymax, chunks


def descriptors(kp, orient, grad, ow, oh, num_dogs, xper, block=1024):
    """desc (n, 128) float64, wm (n,) and valid (n,) (the :49 check; invalid keypoints get zeros)."""
    x, y, s, xi, yi, lev = kp_geom(kp, xper)
    n = len(x)
    valid = (xi >= 0) & (xi < ow) & (yi >= 0) & (yi < oh) & (lev >= 0) & (lev < num_dogs)
    SBP, _, xmin, xmax, ymin, ymax, chunks = desc_window(s, xi, yi, ow, oh)
    th0 = np.asarray(orient, np.float32).reshape(-1, 2)[:, 0].astype(np.float64)
    desc = np.zeros((n, 128))
    wm_out = np.zeros(n)
    for b0 in range(0, n, block):
        sl = np.arange(b0, min(n, b0 + block))
        sl = sl[valid[sl]]
        if not len(sl):
            continue
        S = np.arange(int(chunks[sl].max()) * 256)[None, :]
        c, ty, tx = S >> 8, (S >> 4) & 15, S & 15
        cx, cy = xmin[sl, None] + tx + 16 * c, ymin[sl, None] + ty + 16 * c
        use = (S < 256 * chunks[sl, None]) & (cx <= xmax[sl, None]) & (cy <= ymax[sl, None])
        k, j = np.nonzero(use)
        kk = sl[k]
        px, py = xi[kk] + cx[k, j], yi[kk] + cy[k, j]
        g = grad[lev[kk], py, px].astype(np.float64)
        dx = (px.astype(np.float32) - x[kk]).astype(np.float64)
        dy = (py.astype(np.float32) - y[kk]).astype(np.float64)
        ct, st, sbp = np.cos(th0[kk]), np.sin(th0[kk]), SBP[kk].astype(np.float64)
        nx = (ct * dx + st * dy) / sbp
        ny = (ct * dy - st * dx) / sbp
        nt = 8 * np.mod(g[:, 1] - th0[kk], TWO_PI) / TWO_PI
        wmv = np.exp((nx * nx + ny * ny) / 8) * g[:, 0]
        bx, by, bt = np.floor(nx - 0.5), np.floor(ny - 0.5), np.floor(nt)
        rx, ry, rt = nx - (bx + 0.5), ny - (by + 0.5), nt - bt
        bx, by, bt = bx.astype(np.int64), by.astype(np.int64), bt.astype(np.int64)
        near = np.maximum(np.abs(nx), np.abs(ny)) < 2.5 + 1e-4
        wm_out += np.bincount(kk[near], wmv[near], minlength=n)
        acc = np.zeros(n * 128)
        for dbx in (0, 1):
            for dby in (0, 1):
                ok = (bx + dbx >= -2) & (bx + dbx < 2) & (by + dby >= -2) & (by + dby < 2)
                wxy = wmv * np.abs(1 - dbx - rx) * np.abs(1 - dby - ry)
                for dbt in (0, 1):
                    loc = (bx + dbx + 2) * 8 + (by + dby + 2) * 32 + (bt + dbt) % 8
                    acc += np.bincount(kk[ok] * 128 + loc[ok], (wxy * np.abs(1 - dbt - rt))[ok], minlength=n * 128)
        desc += acc.reshape(n, 128)
    return desc, wm_out, valid
