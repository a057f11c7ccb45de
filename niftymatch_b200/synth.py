"""Deterministic synthetic inputs (SURVEY.md 8d): grayscale scenes in [0,255] and
descriptor sets.  Pure numpy, counter-based splitmix64 so every platform produces the
same bits; no dependence on numpy's Generator streams.

Scene = mid-grey background + K isotropic Gaussian blobs + band-limited texture,
clipped to [0,255] (the range the reference's BGRA->gray conversion produces,
reference src/gpu/kernels/bgra_2_gray.cu:16).  Frame f of a batch uses
seed = 0x5EED0000 + f.
"""
from __future__ import annotations

import numpy as np

SEED_BASE = 0x5EED0000
_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def _splitmix64(x: np.ndarray) -> np.ndarray:
    """splitmix64 finaliser applied to a uint64 counter array."""
    with np.errstate(over="ignore"):
        z = (x + np.uint64(0x9E3779B97F4A7C15)) & _M64
        z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
        z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
        return z ^ (z >> np.uint64(31))


def uniform(seed: int, stream: int, n: int) -> np.ndarray:
    """n float64 uniforms in [0,1) from (seed, stream); counter based."""
    with np.errstate(over="ignore"):
        base = _splitmix64(np.array([seed], dtype=np.uint64) * np.uint64(0x100000001B3)
                           + np.uint64(stream))[0]
        ctr = base + np.arange(n, dtype=np.uint64)
    bits = _splitmix64(ctr) >> np.uint64(11)
    return bits.astype(np.float64) * (1.0 / (1 << 53))


def _blur3(a: np.ndarray) -> np.ndarray:
    """Separable 5-tap binomial-ish blur (sigma ~ 1.0), reflect borders; float64."""
    k = np.array([0.06136, 0.24477, 0.38774, 0.24477, 0.06136])
    p = np.pad(a, ((0, 0), (2, 2)), mode="reflect")
    a = sum(k[i] * p[:, i:i + a.shape[1]] for i in range(5))
    p = np.pad(a, ((2, 2), (0, 0)), mode="reflect")
    return sum(k[i] * p[i:i + a.shape[0], :] for i in range(5))


def scene(width: int, height: int, seed: int, shift=(0.0, 0.0)) -> np.ndarray:
    """One float32 grayscale frame (height, width) in [0,255].

    `shift` = (sx, sy) translates the blob field by a sub-pixel amount so that
    "consecutive" frames contain true correspondences (configs 1 and 5).
    """
    sx, sy = shift
    n_blobs = max(8, (width * height) // 400)
    u = uniform(seed, 1, n_blobs * 4).reshape(n_blobs, 4)
    cx = u[:, 0] * width + sx
    cy = u[:, 1] * height + sy
    sig = 1.5 * np.exp(u[:, 2] * np.log(16.0 / 1.5))
    v = uniform(seed, 2, n_blobs * 2).reshape(n_blobs, 2)
    amp = (8.0 + v[:, 0] * 88.0) * np.where(v[:, 1] < 0.5, -1.0, 1.0)

    img = np.full((height, width), 128.0, dtype=np.float64)
    for i in range(n_blobs):
        r = int(np.ceil(3.5 * sig[i]))
        x0, x1 = max(0, int(cx[i]) - r), min(width, int(cx[i]) + r + 1)
        y0, y1 = max(0, int(cy[i]) - r), min(height, int(cy[i]) + r + 1)
        if x0 >= x1 or y0 >= y1:
            continue
        gx = np.exp(-0.5 * ((np.arange(x0, x1) - cx[i]) / sig[i]) ** 2)
        gy = np.exp(-0.5 * ((np.arange(y0, y1) - cy[i]) / sig[i]) ** 2)
        img[y0:y1, x0:x1] += amp[i] * gy[:, None] * gx[None, :]
    tex = (uniform(seed, 3, width * height).reshape(height, width) - 0.5) * 24.0
    img += _blur3(tex)
    # fresh +-1 sensor noise, different per (seed, shift) so shifted pairs are not copies
    noise_stream = 4 + (int(round(sx * 16)) & 0xFFFF) * 65536 + (int(round(sy * 16)) & 0xFFFF)
    img += (uniform(seed, noise_stream, width * height).reshape(height, width) - 0.5) * 2.0
    return np.clip(img, 0.0, 255.0).astype(np.float32)


def frame_batch(width: int, height: int, n_frames: int, n_scenes: int = 8) -> np.ndarray:
    """(n_frames, height, width) float32.  Frame f = scene (f % n_scenes) translated by a
    per-frame sub-pixel shift (cheap: scenes are rendered once per distinct (scene, shift)
    only when n_frames <= n_scenes; otherwise integer rolls of the base scenes plus fresh
    per-frame noise)."""
    n_scenes = min(n_scenes, n_frames)
    base = [scene(width, height, SEED_BASE + s) for s in range(n_scenes)]
    out = np.empty((n_frames, height, width), dtype=np.float32)
    for f in range(n_frames):
        s, k = f % n_scenes, f // n_scenes
        img = base[s]
        if k:
            img = np.roll(img, (3 * k, 5 * k), axis=(0, 1))
            noise = (uniform(SEED_BASE + f, 9, width * height).reshape(height, width) - 0.5) * 2.0
            img = np.clip(img.astype(np.float64) + noise, 0.0, 255.0).astype(np.float32)
        out[f] = img
    return out


def descriptors(n: int, seed: int, planted_from: np.ndarray | None = None,
                planted_frac: float = 0.2) -> np.ndarray:
    """(n,128) float32 imitating the reference's unnormalised descriptors (SURVEY 8d,
    config 4): 40*|N(0,1)|^3 per element, 60 % of elements zeroed.  With `planted_from`
    (a database), a fraction of rows are copies of random database rows + N(0,2) noise."""
    m = n * 128
    u1 = uniform(seed, 11, m)
    u2 = uniform(seed, 12, m)
    g = np.sqrt(-2.0 * np.log(1.0 - u1)) * np.cos(2.0 * np.pi * u2)
    a = 40.0 * np.abs(g) ** 3
    a[uniform(seed, 13, m) < 0.6] = 0.0
    a = a.reshape(n, 128)
    if planted_from is not None:
        k = int(n * planted_frac)
        rows = (uniform(seed, 14, k) * n).astype(np.int64)
        src = (uniform(seed, 15, k) * planted_from.shape[0]).astype(np.int64)
        w1 = uniform(seed, 16, k * 128)
        w2 = uniform(seed, 17, k * 128)
        noise = 2.0 * np.sqrt(-2.0 * np.log(1.0 - w1)) * np.cos(2.0 * np.pi * w2)
        a[rows] = np.maximum(planted_from[src].astype(np.float64) + noise.reshape(k, 128), 0.0)
    return a.astype(np.float32)


# ---- synthetic registration windows (tests/test_gpu_chain_adjust.py, tools/ransac_report.py --adjust) ----------------
def map_points(G, p):
    """Points p (k, 2) mapped through the 3 x 3 matrix G, in float64."""
    q = np.c_[p, np.ones(len(p))] @ np.asarray(G, np.float64).reshape(3, 3).T
    return q[:, :2] / q[:, 2:]


def camera_chain(kind, n, w, h, seed, step=0.1):
    """Frame k -> frame 0 transforms (n, 3, 3) of a camera path in the family of `kind` (0 translation, 1 similarity,
    2 homography): steps of about step * w px along a slowly turning heading, rotations of up to 0.5 deg, scale changes
    of up to 0.4 % and small perspective terms per frame."""
    rng = np.random.default_rng(seed)
    cx, cy = (w - 1) / 2, (h - 1) / 2
    T = lambda x, y: np.array([[1, 0, x], [0, 1, y], [0, 0, 1.0]])
    G, phi = [np.eye(3)], rng.uniform(0, 2 * np.pi)
    for _ in range(n - 1):
        phi += rng.normal(0, 0.3)
        dd = step * w * rng.uniform(0.6, 1.2)
        M = np.eye(3)
        if kind >= 1:
            a, s = np.deg2rad(rng.uniform(-0.5, 0.5)), 1 + rng.uniform(-0.004, 0.004)
            M = np.array([[s * np.cos(a), -s * np.sin(a), 0], [s * np.sin(a), s * np.cos(a), 0], [0, 0, 1.0]])
        if kind == 2:
            sg = rng.choice([-1, 1])
            M[2, :2] = [sg * 2e-5 * 64 / w, -sg * 2e-5 * 48 / h]
        H = T(cx + dd * np.cos(phi), cy + dd * np.sin(phi)) @ M @ T(-cx, -cy)      # frame k -> frame k + 1
        G.append(G[-1] @ np.linalg.inv(H))
    return np.array(G)


def span_window(kind, n, span, w, h, npts, seed, noise=0.3, outliers=0.3, dtype=np.float32):
    """A window of camera_chain(kind, n, w, h, seed) in the span layout (include/nm_b200.h): for every link (t, t + d) npts
    correspondences, points of frame t that frame t + d also sees, dst with Gaussian noise of `noise` px and a fraction
    `outliers` replaced by random points.  Returns (G, [src_x, src_y, dst_x, dst_y] each (L, npts))."""
    rng = np.random.default_rng(seed + 1000)
    G = camera_chain(kind, n, w, h, seed)
    L = span * n - span * (span + 1) // 2
    arrs = [np.full((L, npts), -1.0, dtype) for _ in range(4)]
    for l, (t, d) in enumerate((t, d) for d in range(1, span + 1) for t in range(n - d)):
        M = np.linalg.inv(G[t + d]) @ G[t]
        src = np.empty((0, 2))
        while len(src) < npts:
            p = rng.uniform([0, 0], [w - 1, h - 1], (4 * npts, 2))
            q = map_points(M, p)
            ok = (q[:, 0] >= 0) & (q[:, 0] <= w - 1) & (q[:, 1] >= 0) & (q[:, 1] <= h - 1)
            src = np.concatenate([src, p[ok]])[:npts]
        dst = map_points(M, src) + rng.normal(0, noise, (npts, 2)) if noise else map_points(M, src)
        bad = rng.random(npts) < outliers
        dst[bad] = rng.uniform([0, 0], [w - 1, h - 1], (bad.sum(), 2))
        for a, v in zip(arrs, (src[:, 0], src[:, 1], dst[:, 0], dst[:, 1])):
            a[l] = v
    return G, arrs
