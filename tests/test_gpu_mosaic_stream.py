"""The mosaic of a frame stream (nm_mosaic_*, niftymatch_b200/mosaic.py): placement against a float64 numpy restatement,
the one-pass blend of a chunk of frames against the per-frame nm_transform_blend_bgra loop on the same textures (bitwise;
that kernel is pinned to the reference by tests/golden/mosaic_128x90.npz), chunking, a registered BGRA stream rendered end
to end, and the argument rules of the entry points."""
import ctypes as C

import numpy as np
import pytest

torch = pytest.importorskip("torch")

from tests._util import _p  # noqa: E402


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    return nm


def _vp(t):
    return C.c_void_p(t.data_ptr())


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def fov_mask(fw, fh):
    """Circular field of view, as a fetoscope's."""
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float64)
    r = 0.49 * min(fw, fh)
    return ((((xx - (fw - 1) / 2) ** 2 + (yy - (fh - 1) / 2) ** 2) < r * r) * 255).astype(np.uint8)


def radial_weights(fw, fh):
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float64)
    d = np.sqrt((xx - (fw - 1) / 2) ** 2 + (yy - (fh - 1) / 2) ** 2) / (0.5 * np.hypot(fw, fh))
    return np.ascontiguousarray(np.maximum(1.0 - d, 0.0) + 1.0 / 64, dtype=np.float32)


def camera_path(n, fw, fh, seed, step=None, deg=0.5, scale=0.004, persp=2e-5):
    """n - 1 pairwise homographies H[p]: frame p -> frame p + 1, a translation of about `step` px along a slowly turning
    heading, a rotation and a scale change about the frame centre and small perspective terms of alternating sign."""
    rng = np.random.default_rng(seed)
    step = step if step is not None else 0.12 * fw
    cx, cy = (fw - 1) / 2, (fh - 1) / 2
    T = lambda x, y: np.array([[1, 0, x], [0, 1, y], [0, 0, 1.0]])
    H, phi = [], rng.uniform(0, 2 * np.pi)
    for p in range(n - 1):
        phi += rng.normal(0, 0.3)
        a = np.deg2rad(rng.uniform(-deg, deg))
        s = 1 + rng.uniform(-scale, scale)
        sg = 1 if p % 2 else -1
        M = np.array([[s * np.cos(a), -s * np.sin(a), 0], [s * np.sin(a), s * np.cos(a), 0],
                      [sg * persp * 64 / fw, -sg * persp * 48 / fh, 1.0]])
        d = step * rng.uniform(0.6, 1.2)
        H.append(T(cx + d * np.cos(phi), cy + d * np.sin(phi)) @ M @ T(-cx, -cy))
    return np.array(H, np.float32).reshape(-1, 9)


def frames_for(n, fw, fh, seed):
    """n BGRA frames with independent channels (smooth, ramp, noise), alpha 255."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float32)
    out = np.empty((n, fh, fw, 4), np.uint8)
    for k in range(n):
        ph = rng.uniform(0, 6.3, 2)
        out[k, ..., 0] = (127 + 110 * np.sin(xx / 5.0 + ph[0]) * np.cos(yy / 4.0 + ph[1])).astype(np.uint8)
        out[k, ..., 1] = ((xx * 3.1 + yy * 1.3 + 17 * k) % 256).astype(np.uint8)
        out[k, ..., 2] = rng.integers(0, 256, (fh, fw), dtype=np.uint8)
        out[k, ..., 3] = 255
    return torch.from_numpy(out).cuda()


def sequential_blend(nm, mosaic, frames, mats, rects, canvas, cwts):
    """The per-frame loop a client drives: one nm_transform_blend_bgra per frame, in order, on the context's textures
    (frame k in slot k: the slots hold what the last Mosaic.blend copied)."""
    lib = nm.load()
    tex, mtex, wtex = mosaic.textures()
    n, fh, fw = frames.shape[:3]
    ch, cw = cwts.shape
    r = rects.cpu().numpy()
    for k in range(n):
        tx, ty, nw, nh = (int(v) for v in r[k])
        assert lib.nm_transform_blend_bgra(_vp(canvas), cw, ch, tex[k], fw, fh, nw, nh, C.c_void_p(mats.data_ptr() + 36 * k), tx, ty,
                                           mtex, _vp(cwts), wtex, _stream()) == 0


def canvas_pair(cw, ch, prefill, seed):
    if prefill:
        g = torch.Generator(device="cpu").manual_seed(seed)
        c = torch.randint(0, 256, (ch, cw, 4), dtype=torch.uint8, generator=g)
        w = torch.rand((ch, cw), generator=g) * 1.75 + 0.25          # every weight non-zero: the weighted branch at once
        c, w = c.cuda(), w.cuda()
    else:
        c = torch.zeros((ch, cw, 4), dtype=torch.uint8, device="cuda")
        w = torch.zeros((ch, cw), dtype=torch.float32, device="cuda")
    return (c.clone(), w.clone()), (c.clone(), w.clone())


def fov_coverage_bounds(mats, rects, cw, ch, fw, fh):
    """Canvas pixels some frame of the chunk blends, bounded from the geometry alone: the mask is the disk of fov_mask,
    sampled bilinearly at texel centres, so a frame position within r - 1 of the centre is inside (all four texels set)
    and one beyond r + 1 is outside.  Returns (lower, upper) pixel counts."""
    r = 0.49 * min(fw, fh)
    cx, cy = (fw - 1) / 2, (fh - 1) / 2
    inner, outer = np.zeros((ch, cw), bool), np.zeros((ch, cw), bool)
    for m, (tx, ty, nw, nh) in zip(np.asarray(mats, np.float64).reshape(-1, 3, 3), rects):
        x0, x1, y0, y1 = max(tx, 0), min(tx + nw, cw), max(ty, 0), min(ty + nh, ch)
        if x0 >= x1 or y0 >= y1:
            continue
        yy, xx = np.mgrid[y0:y1, x0:x1]
        q = m @ np.stack([(xx - tx).ravel(), (yy - ty).ravel(), np.ones(xx.size)])
        d = np.hypot(q[0] / q[2] - cx, q[1] / q[2] - cy).reshape(xx.shape)
        inner[y0:y1, x0:x1] |= d < r - 1
        outer[y0:y1, x0:x1] |= d < r + 1
    return int(inner.sum()), int(outer.sum())


def bitwise_equal(a, b):
    return torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))


@pytest.mark.gpu
@pytest.mark.parametrize("n,fw,fh,max_frames,prefill,crop", [
    (1, 96, 64, 4, False, False),
    (2, 96, 64, 4, True, True),
    (37, 80, 60, 64, False, True),
    (64, 80, 60, 64, True, False),
    (64, 80, 60, 64, False, True),
    (1024, 24, 16, 1024, True, True),
])
def test_stream_blend_equals_per_frame_calls(nm, n, fw, fh, max_frames, prefill, crop):
    """One nm_mosaic_blend_bgra == n nm_transform_blend_bgra calls in frame order, bitwise on canvas bytes and weights.
    Homographies with rotation, scale and perspective; crop = a canvas origin inside the union, so that rects reach
    past every canvas edge with negative tx / ty; canvas sizes that are no multiple of the 64 x 16 tile; one empty rect;
    one rect larger than its footprint (canvas pixels that map beyond fw / fh and beyond -1)."""
    H = camera_path(n, fw, fh, seed=n)
    frames = frames_for(n, fw, fh, seed=n + 1)
    m = nm.Mosaic(fw, fh, max_frames, fov_mask(fw, fh), radial_weights(fw, fh))
    pl = m.place(H)
    ox, oy, bw, bh = pl.bounds.tolist()
    if crop:
        pl = m.place(H, origin=(ox + 13, oy + 7))
        cw, ch = max(bw - 29, 5), max(bh - 19, 3)
    else:
        cw, ch = bw, bh
    if cw % 64 == 0:
        cw -= 1
    if ch % 16 == 0:
        ch -= 1
    rects = pl.rects.clone()
    if n > 2:
        rects[n // 2, 2] = 0                                     # empty
        rects[n // 3, 2:] += torch.tensor([17, 9], dtype=torch.int32, device="cuda")
    fused, seq = canvas_pair(cw, ch, prefill, seed=n + 2)
    m.blend(frames, pl.mats, rects, *fused)
    sequential_blend(nm, m, frames, pl.mats, rects, *seq)
    torch.cuda.synchronize()
    assert bitwise_equal(fused, seq)
    if crop:
        r = rects.cpu().numpy()
        assert (r[:, 0] < 0).any() and (r[:, 1] < 0).any()
        assert (r[:, 0] + r[:, 2] > cw).any() and (r[:, 1] + r[:, 3] > ch).any()
    changed = int((fused[1] != canvas_pair(cw, ch, prefill, seed=n + 2)[0][1]).sum())
    assert changed > 0.2 * fw * fh
    m.close()


@pytest.mark.gpu
def test_chunked_blend_equals_one_call(nm):
    """64 frames as 4 calls of 16 frames = 1 call of 64, bitwise (render_stream's chunking)."""
    n, fw, fh = 64, 112, 72
    H = camera_path(n, fw, fh, seed=3)
    frames = frames_for(n, fw, fh, seed=4)
    mask, wts = fov_mask(fw, fh), radial_weights(fw, fh)
    big, small = nm.Mosaic(fw, fh, 64, mask, wts), nm.Mosaic(fw, fh, 16, mask, wts)
    pl = big.place(H)
    _, _, cw, ch = pl.bounds.tolist()
    one, four = canvas_pair(cw, ch, False, 0)
    big.blend(frames, pl.mats, pl.rects, *one)
    for c0 in range(0, n, 16):
        small.blend(frames[c0:c0 + 16].contiguous(), pl.mats[c0:c0 + 16], pl.rects[c0:c0 + 16], *four)
    c, w, _ = nm.render_stream(frames, torch.from_numpy(H).cuda(), None, mosaic=small)
    torch.cuda.synchronize()
    assert bitwise_equal(one, four) and bitwise_equal(one, (c, w))
    lo, hi = fov_coverage_bounds(pl.mats.cpu().numpy(), pl.rects.cpu().numpy(), cw, ch, fw, fh)
    assert lo > 0.1 * cw * ch and lo <= int((one[1] > 0).sum()) <= hi
    big.close()
    small.close()


# ---- placement: float64 numpy restatement ------------------------------------------------------------------------
def _renorm(a):
    m = np.abs(a).max()
    if not (m > 0) or not np.isfinite(m):
        return a
    return a * np.ldexp(1.0, -int(np.frexp(m)[1]))


def place_ref(H, status, fw, fh, anchor=None, origin=None):
    n = len(H) + 1
    G = np.zeros((n, 3, 3))
    flags = np.zeros(n, np.int32)
    G[0] = _renorm(np.eye(3) if anchor is None else np.asarray(anchor, np.float64).reshape(3, 3))
    for p in range(n - 1):
        h = np.asarray(H[p], np.float64).reshape(3, 3)
        ok = (status is None or status[p][0] != 0) and np.isfinite(h).all()
        if ok:
            ok = abs(np.linalg.det(h)) > 1e-12 * np.abs(h).max() ** 3
        S = np.linalg.inv(h) if ok else np.eye(3)
        flags[p + 1] = 0 if ok else 1
        G[p + 1] = _renorm(G[p] @ S)
    corners = np.array([[-1, -1, 1], [fw, -1, 1], [-1, fh, 1], [fw, fh, 1]], np.float64).T
    rects = np.zeros((n, 4), np.int64)
    for k in range(n):
        q = G[k] @ corners
        with np.errstate(all="ignore"):
            u, v = q[0] / q[2], q[1] / q[2]
        if (q[2] > 0).all() and (np.abs(u) <= 2.0 ** 30).all() and (np.abs(v) <= 2.0 ** 30).all():
            x0, y0 = int(np.floor(u.min())), int(np.floor(v.min()))
            rects[k] = (x0, y0, int(np.ceil(u.max())) - x0 + 1, int(np.ceil(v.max())) - y0 + 1)
        else:
            flags[k] |= 2
    ne = rects[:, 2] > 0
    if origin is not None:
        ox, oy = origin
    else:
        ox, oy = (int(rects[ne, 0].min()), int(rects[ne, 1].min())) if ne.any() else (0, 0)
    bounds = (ox, oy, max(0, int((rects[ne, 0] + rects[ne, 2]).max()) - ox), max(0, int((rects[ne, 1] + rects[ne, 3]).max()) - oy)) \
        if ne.any() else (ox, oy, 0, 0)
    rel = rects.copy()
    rel[ne, 0] -= ox
    rel[ne, 1] -= oy
    mats = np.zeros((n, 9))
    for k in range(n):
        T = np.array([[1, 0, rel[k, 0] + ox], [0, 1, rel[k, 1] + oy], [0, 0, 1.0]])
        mats[k] = _renorm(np.linalg.inv(G[k]) @ T).reshape(9)
    return G.reshape(n, 9), rel, flags, np.array(bounds), mats


def check_placement(pl, ref, fw, fh):
    G, rects, flags, bounds, mats = ref
    g = pl.chain.cpu().numpy()
    assert (np.abs(g - G).max(axis=1) <= 1e-9 * np.abs(G).max(axis=1)).all()
    assert np.array_equal(pl.rects.cpu().numpy(), rects)
    assert np.array_equal(pl.flags.cpu().numpy(), flags)
    assert np.array_equal(pl.bounds.cpu().numpy(), bounds)
    m = pl.mats.cpu().numpy().astype(np.float64)
    ne = rects[:, 2] > 0
    assert (np.abs(m - mats).max(axis=1)[ne] <= 1e-6 * np.abs(mats).max(axis=1)[ne]).all()
    # the one-pixel ring just outside every rect maps (float64) outside the sampling box: nothing the blend would take is cut
    ox, oy = bounds[:2]
    for k in np.nonzero(ne)[0]:
        tx, ty, nw, nh = rects[k]
        xs, ys = np.arange(-1, nw + 1), np.arange(-1, nh + 1)
        ring = np.concatenate([np.stack([xs, np.full_like(xs, -1)]), np.stack([xs, np.full_like(xs, nh)]),
                               np.stack([np.full_like(ys, -1), ys]), np.stack([np.full_like(ys, nw), ys])], axis=1)
        q = np.linalg.inv(G[k].reshape(3, 3)) @ np.stack([ring[0] + tx + ox, ring[1] + ty + oy, np.ones(ring.shape[1])])
        fx, fy = q[0] / q[2], q[1] / q[2]
        assert not ((fx > -1) & (fx < fw) & (fy > -1) & (fy < fh)).any(), k


@pytest.mark.gpu
def test_placement_vs_float64_restatement(nm):
    """Chained transforms to 1e-9, rects / flags / origin / bounds exactly, matrices to float rounding; identity
    substitution (flag bit 0) for a failed status, a singular and a non-finite homography; an anchor; a caller origin."""
    fw, fh, n = 160, 120, 300
    H = camera_path(n, fw, fh, seed=11, persp=4e-5)
    st = np.ones((n - 1, 3), np.int32)
    st[17, 0] = 0
    H[40] = [1, 2, 3, 2, 4, 6, 0, 0, 1]                       # singular
    H[41, 4] = np.nan
    anchor = np.array([0.9, 0.1, 30.0, -0.12, 1.05, -20.0, 1e-6, -2e-6, 1.0], np.float32)
    for an, org in ((None, None), (anchor, None), (anchor, (-50, 37))):
        pl = nm.place(H, st, fw, fh, anchor=an, origin=org)
        ref = place_ref(H, st, fw, fh, an, org)
        check_placement(pl, ref, fw, fh)
        fl = pl.flags.cpu().numpy()
        assert fl[18] == 1 and fl[41] == 1 and fl[42] == 1 and (fl[1:17] == 0).all()
    # a footprint with w <= 0: flag bit 1 and an empty rect; the frames after it keep theirs
    tilt = np.array([1, 0, 0, 0, 1, 0, -0.0045, 0, 1.0], np.float32)        # w = 1 - 0.0045 x (frame 0): <= 0 from x = 223 on
    H2 = camera_path(6, fw, fh, seed=12, persp=0.0)                        # steps of about 19 px
    H2[1] = np.linalg.inv(np.array([[1, 0, 100], [0, 1, 0], [0, 0, 1.0]])).reshape(9)  # frame 2 lies 100 px right of frame 1
    H2[2] = np.array([[1, 0, 100], [0, 1, 0], [0, 0, 1.0]], np.float32).reshape(9)    # and frame 3 back
    pl = nm.place(H2, None, fw, fh, anchor=tilt + np.array([0, 0, 90, 0, 0, 0, 0, 0, 0], np.float32))
    ref = place_ref(H2, None, fw, fh, tilt + np.array([0, 0, 90, 0, 0, 0, 0, 0, 0], np.float32))
    check_placement(pl, ref, fw, fh)
    fl, r = pl.flags.cpu().numpy(), pl.rects.cpu().numpy()
    assert (fl & 2).any() and not (fl & 2).all()
    assert (r[(fl & 2) > 0] == 0).all()


@pytest.mark.gpu
def test_registered_bgra_stream_renders_the_scene(nm):
    """24 integer-offset crops of one scene as BGRA with b = g = r (the grey conversion returns the grey value exactly:
    7 + 72 + 21 = 100), registered by StreamRegistrar on the BGRA chunks and rendered by render_stream: every frame's
    origin within 1 px of the true offset, the canvas within 1 grey level of the scene (median), 8 at the 99th percentile."""
    from niftymatch_b200 import synth
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n = 384, 288, 24
    offs = [(16 + 9 * k + (k % 3), 12 + 5 * k - 2 * (k % 4) + (k // 6)) for k in range(n)]
    W, Hs = max(o[0] for o in offs) + w + 16, max(o[1] for o in offs) + h + 16
    scene = np.rint(synth.scene(W, Hs, synth.SEED_BASE + 21)).astype(np.uint8)
    grey = np.stack([scene[oy: oy + h, ox: ox + w] for ox, oy in offs])
    bgra = np.empty((n, h, w, 4), np.uint8)
    bgra[..., :3] = grey[..., None]
    bgra[..., 3] = 255
    fr = torch.from_numpy(bgra).cuda()
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 8, 8192)
    # the crops move by pure translations, so the translation model: a 4-point homography per pair fits the same
    # correspondences with perspective terms that chain into drift (about 2 px at the centre of frame 23 here)
    reg = StreamRegistrar(sb, chunk=8, kind=nm.TRANSLATION, inlier_threshold=0.25, iterations=512, seed=3)
    H, st = reg.run(lambda t0, t1: fr[t0:t1].contiguous(), 0, n)
    frf = torch.from_numpy(grey.astype(np.float32)).cuda()
    Hf, stf = reg.run(lambda t0, t1: frf[t0:t1].contiguous(), 0, n)
    assert torch.equal(H, Hf) and torch.equal(st, stf)          # BGRA chunks register exactly as their grey frames
    assert (st[:, 0] == 1).all()
    canvas, cwts, pl = nm.render_stream(fr, H, st, fov_mask(w, h), radial_weights(w, h), max_frames=16)
    sb.close()
    # frame k's offset: its centre and its corners mapped into the mosaic (frame 0's coordinates)
    G = pl.chain.cpu().numpy().reshape(n, 3, 3)
    c0, c1 = np.array([(w - 1) / 2, (h - 1) / 2, 1.0]), np.array([[0, 0, 1.0], [w - 1, 0, 1], [0, h - 1, 1], [w - 1, h - 1, 1]]).T
    true = np.array([(ox - offs[0][0], oy - offs[0][1]) for ox, oy in offs], np.float64)
    centre = np.array([(G[k] @ c0)[:2] / (G[k] @ c0)[2] - c0[:2] for k in range(n)])
    corner = max(np.abs((G[k] @ c1)[:2] / (G[k] @ c1)[2] - c1[:2] - true[k][:, None]).max() for k in range(n))
    off_err = np.hypot(*(centre - true).T)
    print(f"frame offsets: max error {off_err.max():.3f} px at the centre, {corner:.3f} px at a corner")
    assert off_err.max() < 1.0 and corner < 1.0, (off_err, corner)
    assert (pl.flags.cpu().numpy() == 0).all()
    bx, by = pl.bounds.tolist()[:2]
    assert (bx, by) == (-1, -1)                                  # the least corner: frame 0's sampling box, exactly
    c, wt = canvas[..., 0].cpu().numpy().astype(np.int32), cwts.cpu().numpy()
    ys, xs = np.nonzero(wt > 0)
    sx, sy = xs + bx + offs[0][0], ys + by + offs[0][1]
    inside = (sx >= 0) & (sx < W) & (sy >= 0) & (sy < Hs)
    assert inside.mean() > 0.999 and inside.sum() > 0.5 * w * h
    err = np.abs(c[ys[inside], xs[inside]] - scene[sy[inside], sx[inside]].astype(np.int32))
    med, p99 = np.median(err), np.percentile(err, 99)
    print(f"render_stream vs scene: median {med}, p99 {p99}, max {err.max()}, {inside.sum()} px")
    assert med <= 1 and p99 <= 8, (med, p99)


@pytest.mark.gpu
def test_mosaic_stream_bad_arguments(nm):
    lib = nm.load()
    fw, fh = 24, 16
    mask, wts = fov_mask(fw, fh), radial_weights(fw, fh)
    ctx = C.c_void_p()
    assert lib.nm_mosaic_create(None, fw, fh, 4, _p(mask), _p(wts)) == -1
    assert lib.nm_mosaic_create(C.byref(ctx), fw, fh, 4, None, _p(wts)) == -1
    assert lib.nm_mosaic_create(C.byref(ctx), fw, fh, 4, _p(mask), None) == -1
    for a, b, mf in ((0, fh, 4), (fw, -1, 4), (fw, fh, 0), (fw, fh, 1025)):
        assert lib.nm_mosaic_create(C.byref(ctx), a, b, mf, _p(mask), _p(wts)) == -1
    assert lib.nm_mosaic_create(C.byref(ctx), fw, fh, 4, _p(mask), _p(wts)) == 0
    fr = torch.zeros((5, fh, fw, 4), dtype=torch.uint8, device="cuda")
    mats = torch.zeros((5, 9), device="cuda")
    rects = torch.zeros((5, 4), dtype=torch.int32, device="cuda")
    cv = torch.zeros((8, 8, 4), dtype=torch.uint8, device="cuda")
    cw = torch.zeros((8, 8), device="cuda")
    s = _stream()
    ok = [ctx, _vp(fr), 4, fw, fh, _vp(mats), _vp(rects), _vp(cv), 8, 8, _vp(cw), s]
    assert lib.nm_mosaic_blend_bgra(*ok) == 0
    for i, bad in ((0, None), (1, None), (5, None), (6, None), (7, None), (10, None), (2, 0), (2, -1), (2, 5), (3, fw - 1),
                   (4, fh + 1), (8, 0), (9, 0)):
        args = list(ok)
        args[i] = bad
        assert lib.nm_mosaic_blend_bgra(*args) == -1, (i, bad)
    H = torch.zeros((4, 9), device="cuda")
    fl, bd = torch.zeros(5, dtype=torch.int32, device="cuda"), torch.zeros(4, dtype=torch.int32, device="cuda")
    pok = [_vp(H), None, 5, fw, fh, None, None, _vp(mats), _vp(rects), _vp(fl), _vp(bd), None, s]
    assert lib.nm_mosaic_place_f32(*pok) == 0
    for i, bad in ((0, None), (2, 0), (3, 0), (4, -2), (7, None), (8, None), (9, None), (10, None)):
        args = list(pok)
        args[i] = bad
        assert lib.nm_mosaic_place_f32(*args) == -1, (i, bad)
    assert lib.nm_mosaic_textures(None, None, None, None) == -1
    torch.cuda.synchronize()
    assert lib.nm_mosaic_destroy(ctx) == 0 and lib.nm_mosaic_destroy(None) == 0


def test_mosaic_create_without_device():
    """No CPU fallback: without a device the context cannot be made."""
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    import niftymatch_b200 as nm
    lib = nm.load()
    mask, wts = fov_mask(24, 16), radial_weights(24, 16)
    ctx = C.c_void_p()
    assert lib.nm_mosaic_create(C.byref(ctx), 24, 16, 4, _p(mask), _p(wts)) == -5      # NM_ERR_NO_DEVICE
    with pytest.raises(nm.NmError):
        nm.Mosaic(24, 16, 4, mask, wts)
