"""Refit of RANSAC models on their inlier sets (nm_ransac_refine_batch_f32, ransac.refine_batch): a float64 numpy
restatement of the three fits (the Levenberg-Marquardt schedule included), checked on exact data without a GPU; on the
GPU the masks against the RANSAC scores, the refits against the restatement, the accuracy gain, determinism, graph
capture, degenerate inputs and the stream pipelines with refinement."""
import ctypes as C

import numpy as np
import pytest

from tests._util import ransac_scene

CORNERS = np.array([[0.0, 0.0], [1919.0, 0.0], [0.0, 1079.0], [1919.0, 1079.0]])


# ---- float64 restatement -----------------------------------------------------------------------------------------
def _hartley(p):
    m = p.mean(0)
    return m, np.sqrt(2.0) / np.sqrt(((p - m) ** 2).sum(1).mean())


def _denormalise(Hn, ms, ss, md, sd):
    Ts = np.array([[ss, 0, -ss * ms[0]], [0, ss, -ss * ms[1]], [0, 0, 1.0]])
    Tdi = np.array([[1 / sd, 0, md[0]], [0, 1 / sd, md[1]], [0, 0, 1.0]])
    H = Tdi @ Hn @ Ts
    return H / H[2, 2]


def fit_translation(s, d):
    t = (d - s).mean(0)
    return np.array([[1, 0, t[0]], [0, 1, t[1]], [0, 0, 1.0]])


def fit_similarity(s, d):
    """[a -b tx; b a ty; 0 0 1], linear least squares in Hartley-normalised coordinates."""
    ms, ss = _hartley(s)
    md, sd = _hartley(d)
    x, y = ((s - ms) * ss).T
    u, v = ((d - md) * sd).T
    one, zero = np.ones_like(x), np.zeros_like(x)
    A = np.concatenate([np.stack([x, -y, one, zero], 1), np.stack([y, x, zero, one], 1)])
    b = np.concatenate([u, v])
    a, bb, tx, ty = np.linalg.solve(A.T @ A, A.T @ b)
    return _denormalise(np.array([[a, -bb, tx], [bb, a, ty], [0, 0, 1.0]]), ms, ss, md, sd)


def _transfer(h, a, b):
    w = h[6] * a + h[7] * b + 1.0
    return (h[0] * a + h[1] * b + h[2]) / w, (h[3] * a + h[4] * b + h[5]) / w, w


def fit_homography(s, d):
    """Normalised DLT (the two rows per point of homography4, eigenvector of the smallest eigenvalue of sum r^T r),
    then Levenberg-Marquardt on the forward transfer error in normalised coordinates: lambda0 = 1e-3 max diag(J^T J),
    (J^T J + lambda diag(J^T J)) delta = -J^T r, accepted -> lambda / 10, rejected -> lambda * 10, at most 20 steps,
    stop when an accepted step gains < 1e-12 of the cost or lambda > 1e16.  None when degenerate."""
    ms, ss = _hartley(s)
    md, sd = _hartley(d)
    a, b = ((s - ms) * ss).T
    u, v = ((d - md) * sd).T
    one, zero = np.ones_like(a), np.zeros_like(a)
    r1 = np.stack([zero, zero, zero, -a, -b, -one, v * a, v * b, v], 1)
    r2 = np.stack([a, b, one, zero, zero, zero, -u * a, -u * b, -u], 1)
    R = np.concatenate([r1, r2])
    ev, V = np.linalg.eigh(R.T @ R)
    if ev[1] <= 1e-12 * ev[-1] or abs(V[8, 0]) <= 1e-12:
        return None
    h = V[:8, 0] / V[8, 0]

    def cost(h):
        X, Y, _ = _transfer(h, a, b)
        return ((X - u) ** 2 + (Y - v) ** 2).sum()

    def normal(h):
        X, Y, w = _transfer(h, a, b)
        Jx = np.stack([a / w, b / w, 1 / w, zero, zero, zero, -a * X / w, -b * X / w], 1)
        Jy = np.stack([zero, zero, zero, a / w, b / w, 1 / w, -a * Y / w, -b * Y / w], 1)
        J = np.concatenate([Jx, Jy])
        r = np.concatenate([X - u, Y - v])
        return J.T @ J, J.T @ r

    c = cost(h)
    JtJ, g = normal(h)
    lam = 1e-3 * JtJ.diagonal().max()
    for _ in range(20):
        try:
            L = np.linalg.cholesky(JtJ + lam * np.diag(JtJ.diagonal()))
            ht = h + np.linalg.solve(L.T, np.linalg.solve(L, -g))
            ct = cost(ht)
        except np.linalg.LinAlgError:
            ct = np.inf
        if ct < c:
            done = c - ct < 1e-12 * c
            h, c, lam = ht, ct, lam * 0.1
            if done:
                break
            JtJ, g = normal(h)
        else:
            lam *= 10.0
            if lam > 1e16:
                break
    return _denormalise(np.append(h, 1.0).reshape(3, 3), ms, ss, md, sd)


FITS = {0: fit_translation, 1: fit_similarity, 2: fit_homography}


def corner_error(H, Ht, corners=CORNERS):
    """Largest and mean distance between the corners mapped by H and by the ground truth Ht."""
    def m(G):
        q = np.asarray(G, np.float64).reshape(3, 3) @ np.c_[corners, np.ones(len(corners))].T
        return (q[:2] / q[2]).T
    e = np.hypot(*(m(H) - m(Ht)).T)
    return e.max(), e.mean()


def true_model(kind, rng):
    if kind == 0:
        return np.array([[1, 0, 12.5], [0, 1, -7.25], [0, 0, 1.0]])
    if kind == 1:
        t, s = 0.05, 1.03
        return np.array([[s * np.cos(t), -s * np.sin(t), 20.0], [s * np.sin(t), s * np.cos(t), -9.0], [0, 0, 1.0]])
    return np.array([[1.02, 0.03, 12.5], [-0.025, 0.99, -7.25], [2.0e-5, -1.5e-5, 1.0]]) + \
        np.diag([1e-3, 1e-3, 0]) * rng.standard_normal()


def scene(Ht, n, rng, outliers=0.3, noise=0.3):
    """n correspondences of Ht in 1920 x 1080 with Gaussian noise, `outliers` of them random.  Returns float32
    src_x, src_y, dst_x, dst_y and the mask of the true inliers."""
    sx, sy = rng.random(n) * 1900 + 10, rng.random(n) * 1060 + 10
    q = Ht @ np.stack([sx, sy, np.ones(n)])
    dx, dy = q[0] / q[2] + rng.normal(0, noise, n), q[1] / q[2] + rng.normal(0, noise, n)
    bad = rng.random(n) < outliers
    dx[bad], dy[bad] = rng.random(bad.sum()) * 1900, rng.random(bad.sum()) * 1060
    return tuple(np.ascontiguousarray(x, np.float32) for x in (sx, sy, dx, dy)) + (~bad,)


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_restatement_recovers_exact_models(kind):
    """On noise-free float64 correspondences every fit returns the true model to 1e-9 relative."""
    rng = np.random.default_rng(40 + kind)
    for trial in range(3):
        Ht = true_model(kind, rng)
        s = np.stack([rng.random(300) * 1900 + 10, rng.random(300) * 1060 + 10], 1)
        q = Ht @ np.c_[s, np.ones(len(s))].T
        d = (q[:2] / q[2]).T
        H = FITS[kind](s, d)
        assert np.abs(H - Ht / Ht[2, 2]).max() <= 1e-9 * np.abs(Ht).max(), (kind, trial, H, Ht)


def test_restatement_degenerate_homographies():
    """Collinear points leave more than one null direction: no homography."""
    k = np.arange(30, dtype=np.float64)
    s = np.stack([100 + 10 * k, 50 + 5 * k], 1)
    assert fit_homography(s, s + [3.0, -2.0]) is None


# ---- the device ----------------------------------------------------------------------------------------------------
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def ragged_batch(n_pairs=16, max_pts=700, seed=30):
    """ransac_scene pairs with ragged counts, one pair with two valid correspondences and one empty pair."""
    arrs = [np.full((n_pairs, max_pts), -1.0, np.float32) for _ in range(4)]
    counts = np.array([max_pts - 37 * p for p in range(n_pairs)], np.int32)
    counts[3], counts[4] = 3, 0
    for p in range(n_pairs):
        sc = ransac_scene(n=max_pts, seed=seed + p)
        for a, v in zip(arrs, sc[:4]):
            a[p, : counts[p]] = v[: counts[p]]
    arrs[0][3, :3] = [5.0, -1.0, 7.0]
    return arrs, counts


def numpy_inliers(H, sx, sy, dx, dy, thr):
    """The inlier rule in float32, and the entries whose squared error is within 1e-4 relative of the threshold."""
    H = H.astype(np.float32)
    with np.errstate(all="ignore"):
        x = H[0] * sx + H[1] * sy + H[2]
        y = H[3] * sx + H[4] * sy + H[5]
        z = H[6] * sx + H[7] * sy + H[8]
        x, y = x / z, y / z
        d2 = (dx - x) * (dx - x) + (dy - y) * (dy - y)
    return (sx >= 0) & (d2 < thr), np.abs(d2 - thr) < 1e-4 * thr


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_mask_is_the_ransac_score(nm, kind):
    """rounds = 0: the mask of every RANSAC model has status[p][1] bits, H comes back bitwise, the mask is the float32
    rule evaluated in numpy (up to entries at the threshold), pairs without a model get {0, 0, 0} and an empty row."""
    arrs, counts = ragged_batch()
    d, cn = [_cu(a) for a in arrs], _cu(counts)
    H, st = nm.ransac_batch(kind, *d, cn, 3.0, 300, seed=77)
    sentinel = torch.full_like(H, 7.0)
    H2, st2, mask = nm.refine_batch(kind, *d, cn, H, st, 3.0, rounds=0, out=(sentinel, torch.full_like(st, 9)))
    H, st, H2, st2, mask = (t.cpu().numpy() for t in (H, st, H2, st2, mask))
    assert np.array_equal(mask.sum(1), st2[:, 1])
    for p in range(len(counts)):
        if st[p, 0] == 0:
            assert st2[p].tolist() == [0, 0, 0] and not mask[p].any() and (H2[p] == 7.0).all(), p
            continue
        assert np.array_equal(H2[p].view(np.int32), H[p].view(np.int32)), p
        assert st2[p].tolist() == [1, st[p, 1], 0], (p, st2[p], st[p])
        ref, near = numpy_inliers(H[p], *(a[p] for a in arrs), 3.0)
        ref[counts[p]:] = False
        assert np.array_equal(mask[p][~near], ref[~near]), p
        assert not mask[p, counts[p]:].any()
    assert (st[:, 0] == 0).sum() >= 1                 # the empty pair (and, for the homography, the two-point pair)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_refit_matches_the_restatement(nm, kind):
    """One refit round on the RANSAC inlier set S0 (the rounds = 0 mask) equals the float64 restatement on S0 to
    < 1e-3 px at the frame corners."""
    rng = np.random.default_rng(60 + kind)
    n_pairs, n = 12, 1500
    arrs = [np.empty((n_pairs, n), np.float32) for _ in range(4)]
    for p in range(n_pairs):
        sc = scene(true_model(kind, rng), n, rng)
        for a, v in zip(arrs, sc[:4]):
            a[p] = v
    d = [_cu(a) for a in arrs]
    H, st = nm.ransac_batch(kind, *d, None, 4.0, 512, seed=5)
    _, _, S0 = nm.refine_batch(kind, *d, None, H, st, 4.0, rounds=0)
    H1, st1, _ = nm.refine_batch(kind, *d, None, H, st, 4.0, rounds=1)
    S0, H1, st1 = S0.cpu().numpy(), H1.cpu().numpy(), st1.cpu().numpy()
    kept = 0
    for p in range(n_pairs):
        if st1[p, 2] == 0:
            continue
        kept += 1
        m = S0[p]
        s = np.stack([arrs[0][p][m], arrs[1][p][m]], 1).astype(np.float64)
        t = np.stack([arrs[2][p][m], arrs[3][p][m]], 1).astype(np.float64)
        emax, _ = corner_error(H1[p], FITS[kind](s, t))
        assert emax < 1e-3, (kind, p, emax)
    assert kept >= n_pairs - 1, st1


@pytest.mark.gpu
def test_refined_homographies_reach_the_noise_floor(nm):
    """Perspective ground truth, sigma = 0.3 px, 30 % outliers, 2 000 correspondences, 64 pairs: the refined corner
    error is at most half the RANSAC model's and within 1.5x the float64 fit to the true inliers; no pair loses
    inliers."""
    rng = np.random.default_rng(8)
    n_pairs, n = 64, 2000
    arrs = [np.empty((n_pairs, n), np.float32) for _ in range(4)]
    truth, floor = [], []
    for p in range(n_pairs):
        Ht = true_model(2, rng)
        sc = scene(Ht, n, rng)
        for a, v in zip(arrs, sc[:4]):
            a[p] = v
        m = sc[4]
        floor.append(corner_error(fit_homography(np.stack([sc[0][m], sc[1][m]], 1).astype(np.float64),
                                                 np.stack([sc[2][m], sc[3][m]], 1).astype(np.float64)), Ht)[1])
        truth.append(Ht)
    d = [_cu(a) for a in arrs]
    H, st = nm.ransac_batch(2, *d, None, 4.0, 1024, seed=1)
    Hr, str_, _ = nm.refine_batch(2, *d, None, H, st, 4.0, rounds=2)
    H, st, Hr, str_ = (t.cpu().numpy() for t in (H, st, Hr, str_))
    e_ransac = np.mean([corner_error(H[p], truth[p])[1] for p in range(n_pairs)])
    e_ref = np.mean([corner_error(Hr[p], truth[p])[1] for p in range(n_pairs)])
    e_floor = np.mean(floor)
    print(f"mean corner error: RANSAC {e_ransac:.4f} px, refined {e_ref:.4f} px, float64 fit to the true inliers "
          f"{e_floor:.4f} px; refits kept {np.bincount(str_[:, 2]).tolist()}")
    assert e_ref <= 0.5 * e_ransac and e_ref <= 1.5 * e_floor, (e_ransac, e_ref, e_floor)
    assert (str_[:, 1] >= st[:, 1]).all() and (str_[:, 0] == 1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_deterministic_batch_independent_in_place_and_graph_capturable(nm, kind):
    rng = np.random.default_rng(90 + kind)
    n_pairs, n = 64, 1200
    arrs = [np.empty((n_pairs, n), np.float32) for _ in range(4)]
    for p in range(n_pairs):
        sc = scene(true_model(kind, rng), n, rng)
        for a, v in zip(arrs, sc[:4]):
            a[p] = v
    counts = rng.integers(n // 2, n + 1, n_pairs).astype(np.int32)
    d, cn = [_cu(a) for a in arrs], _cu(counts)
    H, st = nm.ransac_batch(kind, *d, cn, 4.0, 256, seed=3)
    out = nm.refine_batch(kind, *d, cn, H, st, 4.0, rounds=3)
    again = nm.refine_batch(kind, *d, cn, H, st, 4.0, rounds=3)
    for a, b in zip(out, again):
        assert torch.equal(a, b)
    for p in (0, 17, 63):
        one = nm.refine_batch(kind, *[x[p: p + 1].contiguous() for x in d], cn[p: p + 1].contiguous(), H[p: p + 1].contiguous(),
                              st[p: p + 1].contiguous(), 4.0, rounds=3)
        for a, b in zip(out, one):
            assert torch.equal(a[p: p + 1], b), (kind, p)
    Hi, sti = H.clone(), st.clone()
    res = nm.refine_batch(kind, *d, cn, Hi, sti, 4.0, rounds=3, out=(Hi, sti))
    assert res[0] is Hi and torch.equal(Hi, out[0]) and torch.equal(sti, out[1]) and torch.equal(res[2], out[2])
    # the refine call alone in a CUDA graph, on the RANSAC outputs computed above
    Hg, stg = torch.empty_like(H), torch.empty_like(st)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        nm.refine_batch(kind, *d, cn, H, st, 4.0, rounds=3, out=(Hg, stg))
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    Hg.zero_()
    stg.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        mg = nm.refine_batch(kind, *d, cn, H, st, 4.0, rounds=3, out=(Hg, stg))[2]
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(Hg, out[0]) and torch.equal(stg, out[1]) and torch.equal(mg, out[2])
    if kind == 2:
        assert (out[1][:, 2] >= 1).float().mean() > 0.9


@pytest.mark.gpu
def test_degenerate_inputs_keep_the_model(nm):
    """Exactly four inliers, exactly collinear inliers and a non-finite model come back unchanged with 0 refits kept;
    bad arguments return -1."""
    Ht = np.array([[1.02, 0.03, 12.5], [-0.025, 0.99, -7.25], [2.0e-5, -1.5e-5, 1.0]], np.float32)
    n = 64
    rng = np.random.default_rng(2)
    arrs = [np.full((3, n), -1.0, np.float32) for _ in range(4)]
    # pair 0: four exact inliers (integer source points), the rest far off
    src = np.stack([rng.integers(10, 1900, n), rng.integers(10, 1060, n)], 1).astype(np.float64)
    q = Ht.astype(np.float64) @ np.c_[src, np.ones(n)].T
    dst = (q[:2] / q[2]).T
    dst[4:] += 200.0
    arrs[0][0], arrs[1][0], arrs[2][0], arrs[3][0] = src[:, 0], src[:, 1], dst[:, 0], dst[:, 1]
    # pair 1: 30 collinear integer points, translated by an integer vector
    k = np.arange(30)
    arrs[0][1, :30], arrs[1][1, :30] = 100 + 10 * k, 50 + 5 * k
    arrs[2][1, :30], arrs[3][1, :30] = 103 + 10 * k, 48 + 5 * k
    # pair 2: pair 0's points, model NaN
    for a in arrs:
        a[2] = a[0]
    H = np.stack([Ht.reshape(-1), np.array([1, 0, 3, 0, 1, -2, 0, 0, 1], np.float32), np.full(9, np.nan, np.float32)])
    st = np.array([[1, 4, 0], [1, 30, 0], [1, 0, 0]], np.int32)
    d = [_cu(a) for a in arrs]
    Hd = _cu(H)
    Ho, sto, mask = nm.refine_batch(2, *d, None, Hd, _cu(st), 4.0, rounds=2)
    Ho, sto, mask = Ho.cpu().numpy(), sto.cpu().numpy(), mask.cpu().numpy()
    _, st0, _ = nm.refine_batch(2, *d, None, Hd, _cu(st), 4.0, rounds=0)
    assert np.array_equal(Ho.view(np.int32), H.view(np.int32))
    assert sto.tolist() == st0.cpu().numpy().tolist() and sto[:, 2].tolist() == [0, 0, 0], sto
    assert sto[0, 1] == 4 and sto[1, 1] == 30 and sto[2, 1] == 0
    assert mask[0, :4].all() and not mask[0, 4:].any() and not mask[2].any()
    # the same pairs through the translation and similarity fits are not degenerate
    for kind in (0, 1):
        Hk, stk, _ = nm.refine_batch(kind, *[a[1:2].contiguous() for a in d], None, Hd[1:2].contiguous(),
                                     _cu(st[1:2]), 4.0, rounds=2)
        assert stk.cpu().tolist()[0][1] == 30
    # argument checks of nm_ransac_refine_batch_f32
    lib = nm.load()
    p = lambda t: C.c_void_p(t.data_ptr())
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    Hout, sout = torch.empty(3, 9, device="cuda"), torch.empty(3, 3, dtype=torch.int32, device="cuda")
    good = dict(kind=2, stride=n, max_pts=n, n_pairs=3, rounds=1)

    def call(kind=2, stride=n, max_pts=n, n_pairs=3, rounds=1, sx=p(d[0]), Hin=p(Hd), Hout_=p(Hout), sout_=p(sout)):
        return lib.nm_ransac_refine_batch_f32(kind, sx, p(d[1]), p(d[2]), p(d[3]), stride, None, max_pts, n_pairs, 4.0,
                                              Hin, None, rounds, Hout_, sout_, None, s)
    assert call(**good) == 0
    for bad in (dict(kind=3), dict(kind=-1), dict(rounds=-1), dict(n_pairs=0), dict(max_pts=0), dict(stride=-1),
                dict(sx=None), dict(Hin=None), dict(Hout_=None), dict(sout_=None)):
        assert call(**bad) == -1, bad
    torch.cuda.synchronize()


# ---- the stream pipelines ------------------------------------------------------------------------------------------
def _crop_stream():
    from niftymatch_b200 import synth
    w, h, n = 384, 288, 24
    offs = [(16 + 9 * k + (k % 3), 12 + 5 * k - 2 * (k % 4) + (k // 6)) for k in range(n)]
    W, Hs = max(o[0] for o in offs) + w + 16, max(o[1] for o in offs) + h + 16
    scene_ = np.rint(synth.scene(W, Hs, synth.SEED_BASE + 21)).astype(np.uint8)
    grey = np.stack([scene_[oy: oy + h, ox: ox + w] for ox, oy in offs])
    bgra = np.empty((n, h, w, 4), np.uint8)
    bgra[..., :3] = grey[..., None]
    bgra[..., 3] = 255
    return w, h, n, offs, bgra


@pytest.mark.gpu
def test_refined_homography_stream_drifts_less(nm):
    """The crop stream of test_registered_bgra_stream_renders_the_scene registered with the HOMOGRAPHY model at its
    0.5 px threshold: with two refit rounds the chained corners drift less than without.  On these SIFT correspondences
    a least-squares refit often counts a few inliers fewer than the count-maximising 4-point model and is then not kept
    (9 of 23 pairs keep one; about 3 px at the worst corner against 4.7 px unrefined), so the chain does not reach the
    1 px of the translation model."""
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n, offs, bgra = _crop_stream()
    fr = torch.from_numpy(bgra).cuda()
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 8, 8192)
    c0, c1 = np.array([(w - 1) / 2, (h - 1) / 2, 1.0]), np.array([[0, 0, 1.0], [w - 1, 0, 1], [0, h - 1, 1], [w - 1, h - 1, 1]]).T
    true = np.array([(ox - offs[0][0], oy - offs[0][1]) for ox, oy in offs], np.float64)
    errs, kept = {}, None
    for rounds in (0, 2):
        reg = StreamRegistrar(sb, chunk=8, kind=nm.HOMOGRAPHY, inlier_threshold=0.25, iterations=512, seed=3,
                              refine_rounds=rounds)
        H, st = reg.run(lambda t0, t1: fr[t0:t1].contiguous(), 0, n)
        assert (st[:, 0] == 1).all()
        G = nm.place(H, st, w, h).chain.cpu().numpy().reshape(n, 3, 3)
        centre = np.array([(G[k] @ c0)[:2] / (G[k] @ c0)[2] - c0[:2] for k in range(n)])
        corner = max(np.abs((G[k] @ c1)[:2] / (G[k] @ c1)[2] - c1[:2] - true[k][:, None]).max() for k in range(n))
        errs[rounds] = (np.hypot(*(centre - true).T).max(), corner)
        if rounds:
            kept = st[:, 2].cpu().numpy()
        print(f"homography stream, refine_rounds {rounds}: max error {errs[rounds][0]:.3f} px at the centre, "
              f"{corner:.3f} px at a corner")
    sb.close()
    print("refits kept per pair:", kept.tolist())
    assert (kept >= 1).sum() >= 5, kept
    assert errs[2][1] < errs[0][1] and errs[2][0] < 1.0, errs


@pytest.mark.gpu
def test_stream_registrar_with_refinement_equals_register_stream(nm):
    """The 9-frame stream of test_stream_registrar_device_pipeline_equals_the_per_pair_path: with refinement,
    StreamRegistrar equals register_stream bitwise at chunk sizes 5, 3, 2 and over 2- and 3-rank shardings; with
    refine_rounds = 0 it equals the unrefined register_stream.  Refinement never lowers an inlier count."""
    from niftymatch_b200 import synth
    from niftymatch_b200.dist import StreamRegistrar, frame_range
    w, h = 512, 384
    base = synth.scene(w + 64, h + 64, synth.SEED_BASE + 9)
    offs = [(8, 8), (12, 10), (18, 9), (20, 16), (27, 20), (30, 26), (38, 30), (40, 35), (44, 41)]
    fr = _cu(np.stack([base[oy: oy + h, ox: ox + w] for ox, oy in offs]))
    n = len(offs)
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 5, 8192)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    n_kept = 0
    for thr in (1.0, 0.25):                   # 1.0: the unrefined test's threshold; 0.25 keeps more of the refits
        kw = dict(kind=nm.HOMOGRAPHY, inlier_threshold=thr, iterations=512, seed=5)
        _, H0, s0 = nm.register_stream(sb, fr, chunk=4, **kw)
        _, Href, sref = nm.register_stream(sb, fr, chunk=4, refine_rounds=2, **kw)
        H0, s0, Href, sref = (t.cpu().numpy() for t in (H0, s0, Href, sref))
        assert (sref[:, 0] == 1).all() and (sref[:, 1] >= s0[:, 1]).all(), (s0, sref)
        n_kept += int((sref[:, 2] >= 1).sum())
        print(f"threshold {thr}: refits kept {sref[:, 2].tolist()}")
        H, st = StreamRegistrar(sb, chunk=4, **kw).run(frames_of, 0, n)
        assert np.array_equal(H.cpu().numpy(), H0) and np.array_equal(st.cpu().numpy(), s0)
        for chunk in (5, 3, 2):
            H, st = StreamRegistrar(sb, chunk=chunk, refine_rounds=2, **kw).run(frames_of, 0, n)
            assert np.array_equal(H.cpu().numpy(), Href) and np.array_equal(st.cpu().numpy(), sref), (thr, chunk)
        reg = StreamRegistrar(sb, chunk=4, refine_rounds=2, **kw)
        for world in (2, 3):
            got = [reg.run(frames_of, *frame_range(n, world, rank, overlap=1)) for rank in range(world)]
            assert np.array_equal(np.concatenate([g[0].cpu().numpy() for g in got]), Href), (thr, world)
            assert np.array_equal(np.concatenate([g[1].cpu().numpy() for g in got]), sref), (thr, world)
    sb.close()
    assert n_kept >= 1
