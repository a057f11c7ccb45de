"""Test-side bindings of the CHECKERS: the CPU oracle (oracle/libnm_oracle.so) and the
reference's own CUDA build (oracle/_ref/libnmref.so).  Both export the same frame-level
entry point, so one wrapper serves both.  Test infrastructure only."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_SO = os.path.join(ROOT, "oracle", "libnm_oracle.so")
REF_SO = os.path.join(ROOT, "oracle", "_ref", "libnmref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def octave_dims(w, h, n_oct):
    return [(w >> o, h >> o) for o in range(n_oct)]


class FrameChecker:
    """sift_frame / match on host arrays through `<prefix>_sift_frame`, `<prefix>_match`."""

    def __init__(self, lib, prefix):
        self.lib, self.prefix = lib, prefix
        self._frame = getattr(lib, prefix + "_sift_frame")
        self._frame.restype = C.c_int
        self._frame_masked = getattr(lib, prefix + "_sift_frame_masked", None)
        if self._frame_masked is not None:
            self._frame_masked.restype = C.c_int
        self._match = getattr(lib, prefix + "_match")
        self._match.restype = C.c_int

    def sift_frame(self, image, peak=0.0, edge=-1.0, num_octaves=-1, capacity=65536, clear_grad=1,
                   kp_cap=200000, want_levels=True, want_grad=False, orient_mode=None, orient_in=None, mask=None):
        """orient_mode: 0 = public-API orientation semantics (window clamp 10; the reference's
        own kernel deadlocks on sm_70+, so the reference build refuses it), 1 = arithmetic of the
        reference's kernel_orientations_naive (no clamp), 2 = injected orientations.
        Default: 0 for the CPU oracle, 1 for the reference build.
        mask: optional h x w float image -> the masked detector (compute_keypoints_with_mask)."""
        if orient_mode is None:
            orient_mode = 0 if self.prefix == "orc" else 1
        if orient_in is not None:
            orient_in = np.ascontiguousarray(orient_in, dtype=np.float32)
        h, w = image.shape
        image = np.ascontiguousarray(image, dtype=np.float32)
        cfg = np.array([peak, edge, num_octaves, capacity, clear_grad, orient_mode], dtype=np.float32)
        desc = np.zeros((capacity, 128), np.float32)
        x = np.zeros(capacity, np.float32)
        y = np.zeros(capacity, np.float32)
        n = C.c_int()
        max_oct = 12
        tot = sum((w >> o) * (h >> o) for o in range(max_oct))
        levels = np.zeros(tot * 6, np.float32) if want_levels else None
        grad = np.zeros(tot * 3 * 2, np.float32) if want_grad else None
        kpts = np.zeros((kp_cap, 4), np.float32)
        orient = np.zeros((kp_cap, 2), np.float32)
        seg = np.zeros(max_oct * 3, np.int32)
        if mask is None:
            n_oct = self._frame(_p(image), w, h, _p(cfg), _p(desc), _p(x), _p(y), C.byref(n), _p(levels), _p(kpts),
                                _p(orient), _p(seg), kp_cap, _p(grad), _p(orient_in))
        else:
            mask = np.ascontiguousarray(mask, dtype=np.float32)
            assert mask.shape == (h, w) and self._frame_masked is not None
            n_oct = self._frame_masked(_p(image), w, h, _p(cfg), _p(desc), _p(x), _p(y), C.byref(n), _p(levels),
                                       _p(kpts), _p(orient), _p(seg), kp_cap, _p(grad), _p(orient_in), _p(mask))
        if n_oct < 0:
            raise RuntimeError(f"{self.prefix}_sift_frame refused (code {n_oct}): orient_mode {orient_mode}")
        out = {"n_oct": n_oct, "n": n.value, "desc": desc[: n.value], "x": x[: n.value], "y": y[: n.value],
               "seg_counts": seg[: n_oct * 3].copy()}
        nk = int(seg[: n_oct * 3].sum())
        out["kpts"], out["orient"] = kpts[:nk], orient[:nk]
        if want_levels:
            lv, off = [], 0
            for (ow, oh) in octave_dims(w, h, n_oct):
                lv.append([levels[off + i * ow * oh: off + (i + 1) * ow * oh].reshape(oh, ow) for i in range(6)])
                off += 6 * ow * oh
            out["levels"] = lv
        if want_grad:
            gr, off = [], 0
            for (ow, oh) in octave_dims(w, h, n_oct):
                gr.append(grad[off: off + 6 * ow * oh].reshape(3, oh, ow, 2))
                off += 6 * ow * oh
            out["grad"] = gr
        return out

    def match(self, A, B, ambiguity=0.8, match_io=None, want_distance=False):
        A = np.ascontiguousarray(A, np.float32)
        B = np.ascontiguousarray(B, np.float32)
        nA, nB = A.shape[0], B.shape[0]
        m = np.full(nA, -1, np.int32) if match_io is None else np.ascontiguousarray(match_io, np.int32).copy()
        if self.prefix == "orc":
            self._match(_p(A), nA, _p(B), nB, C.c_float(ambiguity), _p(m))
            if want_distance:
                D = np.zeros((nA, nB), np.float32)
                self.lib.orc_dist2(_p(A), nA, _p(B), nB, 128, _p(D))
                return m, D
            return m
        D = np.zeros((nA, nB), np.float32) if want_distance else None
        self._match(_p(A), nA, _p(B), nB, C.c_float(ambiguity), _p(m), _p(D))
        return (m, D) if want_distance else m


# ---- registration (align_points / RANSAC) checkers: oracle (orc_*) and reference (nmref_*) -------
def ransac_scene(n=400, seed=7, outliers=0.3, invalid=0.1, noise=0.3):
    """Correspondences under a known homography: `outliers` of them wrong, `invalid` marked -1 (unmatched),
    Gaussian noise on the rest.  Returns src_x, src_y, dst_x, dst_y (float32) and the 3x3 ground truth."""
    rng = np.random.default_rng(seed)
    Ht = np.array([[1.02, 0.03, 12.5], [-0.025, 0.99, -7.25], [2.0e-5, -1.5e-5, 1.0]])
    sx = rng.random(n) * 1900 + 10
    sy = rng.random(n) * 1060 + 10
    q = Ht @ np.stack([sx, sy, np.ones(n)])
    dx = q[0] / q[2] + rng.normal(0, noise, n)
    dy = q[1] / q[2] + rng.normal(0, noise, n)
    bad = rng.random(n) < outliers
    dx[bad] = rng.random(bad.sum()) * 1900
    dy[bad] = rng.random(bad.sum()) * 1060
    inv = rng.random(n) < invalid
    sx[inv] = sy[inv] = dx[inv] = dy[inv] = -1.0
    return tuple(np.ascontiguousarray(a, np.float32) for a in (sx, sy, dx, dy)) + (Ht,)


def ransac_rand_lists(sx, iterations=192, seed=11):
    """Index lists (valid correspondences only, like ransac.cu:533-555) for the three estimators, with
    repeated-index iterations planted (they must score 0 with H = 0)."""
    rng = np.random.default_rng(seed)
    valid = np.nonzero(sx >= 0)[0]
    out = {}
    for kind, m in ((0, 1), (1, 2), (2, 4)):
        rl = valid[rng.integers(0, len(valid), size=(iterations, m))].astype(np.int32)
        if m > 1:
            rl[5, 1] = rl[5, 0]
            rl[17, m - 1] = rl[17, 0]
        out[kind] = np.ascontiguousarray(rl.reshape(-1))
    return out


def checker_ransac_hypotheses(lib, prefix, kind, sx, sy, dx, dy, rand_list, thr):
    m = (1, 2, 4)[kind]
    it = len(rand_list) // m
    H = np.zeros((it, 9), np.float32)
    inl = np.zeros(it, np.int32)
    fn = getattr(lib, prefix + "_ransac_hypotheses")
    fn.restype = C.c_int
    rc = fn(kind, _p(sx), _p(sy), _p(dx), _p(dy), len(sx), _p(rand_list), it, C.c_float(thr), _p(H), _p(inl))
    assert not rc, rc
    return H, inl


def normalise_h(H):
    """Homographies up to scale: divide by the Frobenius norm, sign of the largest element positive."""
    H = np.asarray(H, np.float64).reshape(-1, 9)
    nrm = np.linalg.norm(H, axis=1, keepdims=True)
    nrm[nrm == 0] = 1.0
    return H / nrm


# ---- input preprocessing checkers -----------------------------------------------------------------
def preprocess_inputs(seed=5):
    """Small deterministic inputs of the rank-2 functions: a BGRA frame, a float image with values around and
    beyond the byte range, coordinate maps with a camera model."""
    rng = np.random.default_rng(seed)
    h, w = 96, 160
    bgra = rng.integers(0, 256, (h, w, 4), dtype=np.uint8)
    fimg = (rng.random((h, w)) * 300 - 20).astype(np.float32)
    fimg[0, :8] = [0.0, 0.999, 1.0, 254.999, 255.0, 255.5, 256.0, 1000.0]
    fimg[1, :6] = [-0.5, -1.0, -300.0, 511.7, 65536.0, 3.0e9]
    yy, xx = np.mgrid[0:h, 0:w].astype(np.float32)
    cam = np.array([140.0, 150.0, 79.5, 47.5], np.float32)        # fx, fy, cx, cy
    dist = np.array([-0.21, 0.06, -0.004], np.float32)            # k1, k2, k3
    gray8 = rng.integers(0, 256, (h, w), dtype=np.uint8)
    return dict(bgra=bgra, fimg=fimg, x=np.ascontiguousarray(xx), y=np.ascontiguousarray(yy), cam=cam, dist=dist, gray8=gray8)


def all_bgr_words():
    """Every (b, g, r) combination once, alpha = low byte of the index: 4096 x 4096 BGRA pixels."""
    i = np.arange(1 << 24, dtype=np.uint32)
    px = np.empty((1 << 24, 4), np.uint8)
    px[:, 0] = i & 255
    px[:, 1] = (i >> 8) & 255
    px[:, 2] = (i >> 16) & 255
    px[:, 3] = (i * 7) & 255
    return px.reshape(4096, 4096, 4)


def gray_double_formula(bgra):
    """(float)(0.07*b + 0.72*g + 0.21*r) in double, the expression of bgra_2_gray.cu:16."""
    b = bgra[..., 0].astype(np.float64)
    g = bgra[..., 1].astype(np.float64)
    r = bgra[..., 2].astype(np.float64)
    return (0.07 * b + 0.72 * g + 0.21 * r).astype(np.float32)


def mosaic_inputs(seed=6):
    """A smooth BGRA frame (so that one-LSB filtering differences stay one LSB), a circular byte mask, a
    distance-to-border weight map, perspective matrices and canvas offsets for three blended warps."""
    rng = np.random.default_rng(seed)
    fh, fw = 90, 128
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float32)
    frame = np.zeros((fh, fw, 4), np.uint8)
    frame[..., 0] = (127 + 100 * np.sin(xx / 9.0) * np.cos(yy / 7.0)).astype(np.uint8)
    frame[..., 1] = (xx * 1.7 + yy * 0.4).astype(np.uint8)
    frame[..., 2] = rng.integers(0, 256, (fh, fw)).astype(np.uint8)
    frame[..., 3] = 255
    mask = (((xx - fw / 2) ** 2 + (yy - fh / 2) ** 2) < (0.47 * fh) ** 2).astype(np.uint8) * 255
    wts = np.minimum(np.minimum(xx + 1, fw - xx), np.minimum(yy + 1, fh - yy)).astype(np.float32) / 16.0
    mats = np.array([[1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0],
                     [0.98, 0.05, -3.2, -0.04, 1.01, 2.6, 1.0e-4, -2.0e-4, 1.0],
                     [1.03, -0.02, 5.5, 0.03, 0.97, -4.25, -1.5e-4, 1.0e-4, 1.0]], np.float32)
    tx = np.array([10, 22, -6], np.int32)
    ty = np.array([8, -5, 30], np.int32)
    return dict(frame=frame, mask=mask, wts=np.ascontiguousarray(wts), mats=mats, tx=tx, ty=ty)


def load_oracle():
    if not os.path.exists(ORACLE_SO) or os.path.getmtime(ORACLE_SO) < os.path.getmtime(os.path.join(ROOT, "oracle", "nm_oracle.c")):
        subprocess.check_call(["make", "-C", ROOT, "oracle/libnm_oracle.so"], stdout=subprocess.DEVNULL)
    return FrameChecker(C.CDLL(ORACLE_SO), "orc")


def orc_orientations(lib, kp, grad, xper=1.0):
    """orc_orientations (public-API semantics, window clamp 10) on a (levels, oh, ow, 2) gradient buffer."""
    kp, grad = np.ascontiguousarray(kp, np.float32), np.ascontiguousarray(grad, np.float32)
    res = np.full((len(kp), 2), -1, np.float32)
    lib.orc_orientations(_p(kp), _p(grad), len(kp), grad.shape[2], grad.shape[1], C.c_float(1.5), C.c_float(xper),
                         _p(res), 10)
    return res


def orc_descriptors(lib, kp, orient, grad, num_dogs=3, xper=1.0):
    """orc_descriptors on a (levels, oh, ow, 2) gradient buffer: desc (n, 128), x, y (zeros where :49 fails)."""
    kp, grad = np.ascontiguousarray(kp, np.float32), np.ascontiguousarray(grad, np.float32)
    orient = np.ascontiguousarray(orient, np.float32)
    n = len(kp)
    desc, x, y = np.zeros((n, 128), np.float32), np.zeros(n, np.float32), np.zeros(n, np.float32)
    lib.orc_descriptors(_p(kp), _p(orient), _p(grad), n, grad.shape[2], grad.shape[1], num_dogs, C.c_float(xper),
                        _p(desc), _p(x), _p(y))
    return desc, x, y


def load_reflib():
    if not os.path.exists(REF_SO):
        return None
    return FrameChecker(C.CDLL(REF_SO), "nmref")


# ---- comparison helpers shared by the CPU and GPU parity tests -------------------------
def match_keypoints(kp_a, kp_b, tol=0.01):
    """Greedy one-to-one association of float4 keypoints (x, y, sigma, level) by level and
    position (<= tol px).  Returns index arrays (ia, ib)."""
    ia, ib = [], []
    used = np.zeros(len(kp_b), bool)
    for i, k in enumerate(kp_a):
        cand = np.where((kp_b[:, 3] == k[3]) & ~used & (np.abs(kp_b[:, 0] - k[0]) <= tol) & (np.abs(kp_b[:, 1] - k[1]) <= tol))[0]
        if len(cand):
            j = cand[np.argmin(np.abs(kp_b[cand, 0] - k[0]) + np.abs(kp_b[cand, 1] - k[1]))]
            used[j] = True
            ia.append(i)
            ib.append(j)
    return np.array(ia, int), np.array(ib, int)


def equal_at_stored(level, stored):
    """Bitwise equality with a golden level at the pixels the fixture keeps: large levels are stored at a fixed sample
    of their pixels, NaN elsewhere (tests/golden/make_golden.py, sample_level).  A computed level holds no NaN."""
    keep = ~np.isnan(stored)
    return level.shape == stored.shape and not np.isnan(level).any() and np.array_equal(level[keep], stored[keep])


def ang_diff(a, b):
    d = np.abs(a - b)
    return np.minimum(d, np.abs(2 * np.pi - d))
