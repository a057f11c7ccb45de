"""Joint adjustment of a window's chain from skip links (nm_match_pairs_span_f32, nm_align_pairs_span_f32,
nm_ransac_adjust_chain_f32, StreamRegistrar(span > 1)).

A float64 numpy restatement of the adjustment (same initial poses, parameterisation, cost and Levenberg-Marquardt
schedule) is checked without a GPU: it recovers exact chains from noise-free correspondences and reaches the minimum
scipy.optimize.least_squares finds.  The GPU tests compare the device with it and with the existing per-pair paths."""
import ctypes as C

import numpy as np
import pytest
import torch

# ---- the restatement ------------------------------------------------------------------------------------------------
NPAR = {0: 2, 1: 4, 2: 8}
MINPTS = {0: 1, 1: 2, 2: 4}


def n_links(n, span):
    return span * n - span * (span + 1) // 2


def link_row(n, t, d):
    return (d - 1) * n - (d - 1) * d // 2 + t


def links(n, span):
    return [(t, d) for d in range(1, span + 1) for t in range(n - d)]


def _chain_step(H):
    """nm_chain_step: H^-1 in float64, the identity for a non-finite or singular model."""
    h = np.asarray(H, np.float64).reshape(3, 3)
    if not np.isfinite(h).all():
        return np.eye(3)
    a = h.reshape(-1)
    det = a[0] * (a[4] * a[8] - a[5] * a[7]) - a[1] * (a[3] * a[8] - a[5] * a[6]) + a[2] * (a[3] * a[7] - a[4] * a[6])
    m = np.abs(a).max()
    if not abs(det) > 1e-12 * m ** 3:
        return np.eye(3)
    return np.linalg.inv(h)


def _renormalise(g):
    m = np.abs(g).max()
    if m > 0 and np.isfinite(m):
        g = g * 2.0 ** -np.frexp(m)[1]
    return g


def geometry(w, h):
    """N: centre the frame, scale by 2 / max(w, h)."""
    s = 2.0 / max(w, h)
    cx, cy = 0.5 * (w - 1), 0.5 * (h - 1)
    return np.array([[s, 0, -s * cx], [0, s, -s * cy], [0, 0, 1.0]])


def matrix(kind, th):
    if kind == 0:
        return np.array([[1, 0, th[0]], [0, 1, th[1]], [0, 0, 1.0]])
    if kind == 1:
        return np.array([[th[0], -th[1], th[2]], [th[1], th[0], th[3]], [0, 0, 1.0]])
    return np.append(th, 1.0).reshape(3, 3)


def params(kind, G):
    G = G / G[2, 2]
    if kind == 0:
        return np.array([G[0, 2], G[1, 2]])
    if kind == 1:
        return np.array([G[0, 0], G[1, 0], G[0, 2], G[1, 2]])
    return G.reshape(-1)[:8].copy()


def project(kind, th, p):
    """pi(Gn(th) p) for points p (k, 2) and the derivatives (k, 2, P) with respect to th."""
    x, y = p[:, 0], p[:, 1]
    k = len(p)
    J = np.zeros((k, 2, NPAR[kind]))
    if kind == 0:
        U, V = x + th[0], y + th[1]
        J[:, 0, 0] = J[:, 1, 1] = 1.0
    elif kind == 1:
        U = th[0] * x - th[1] * y + th[2]
        V = th[1] * x + th[0] * y + th[3]
        J[:, 0] = np.stack([x, -y, np.ones(k), np.zeros(k)], 1)
        J[:, 1] = np.stack([y, x, np.zeros(k), np.ones(k)], 1)
    else:
        iw = 1.0 / (th[6] * x + th[7] * y + 1.0)
        U = (th[0] * x + th[1] * y + th[2]) * iw
        V = (th[3] * x + th[4] * y + th[5]) * iw
        a, b, z = x * iw, y * iw, np.zeros(k)
        J[:, 0] = np.stack([a, b, iw, z, z, z, -U * a, -U * b], 1)
        J[:, 1] = np.stack([z, z, z, a, b, iw, -V * a, -V * b], 1)
    return np.stack([U, V], 1), J


class Window:
    """The links of one window in the span layout: per link the normalised mask points (a in frame t, b in frame t + d)."""

    def __init__(self, kind, n, span, w, h, sx, sy, dx, dy, counts, masks, H, status):
        self.kind, self.n, self.span, self.P = kind, n, span, NPAR[kind]
        self.N = geometry(w, h)
        self.s = self.N[0, 0]
        L = n_links(n, span)
        H = np.asarray(H).reshape(L, 9)
        status = np.asarray(status).reshape(L, 3)
        self.pts = []
        for l in range(L):
            c = sx.shape[1] if counts is None else min(int(counts[l]), sx.shape[1])
            m = np.asarray(masks[l][:c], bool)
            a = np.stack([sx[l][:c][m], sy[l][:c][m]], 1).astype(np.float64)
            b = np.stack([dx[l][:c][m], dy[l][:c][m]], 1).astype(np.float64)
            self.pts.append(((a - [0.5 * (w - 1), 0.5 * (h - 1)]) * self.s, (b - [0.5 * (w - 1), 0.5 * (h - 1)]) * self.s))
        usable = [status[l, 0] == 1 and len(self.pts[l][0]) >= MINPTS[kind] for l in range(L)]
        # initial poses: place_kernel's chain over the smallest usable d
        G = [np.eye(3)]
        self.conn = [True]
        for k in range(1, n):
            for d in range(1, min(span, k) + 1):
                l = link_row(n, k - d, d)
                if self.conn[k - d] and usable[l]:
                    G.append(_renormalise(G[k - d] @ _chain_step(H[l])))
                    self.conn.append(True)
                    break
            else:
                G.append(G[k - 1].copy())
                self.conn.append(False)
        self.x0 = np.array([params(kind, self.N @ g @ np.linalg.inv(self.N)) for g in G])
        self.x0[0] = params(kind, np.eye(3))
        self.used = [usable[link_row(n, t, d)] and self.conn[t] and self.conn[t + d] for t, d in links(n, span)]
        self.order = links(n, span)
        self.free = [k for k in range(1, n) if self.conn[k]]

    def residuals(self, x):
        out = []
        for (t, d), u, (a, b) in zip(self.order, self.used, self.pts):
            if u:
                out.append(project(self.kind, x[t], a)[0] - project(self.kind, x[t + d], b)[0])
        return np.concatenate(out) if out else np.zeros((0, 2))

    def system(self, x):
        """cost, J^T J and J^T r over the free frames (normalised units)."""
        P, col = self.P, {k: i for i, k in enumerate(self.free)}
        A = np.zeros((len(self.free) * P,) * 2)
        g = np.zeros(len(self.free) * P)
        cost = 0.0
        for (t, d), u, (a, b) in zip(self.order, self.used, self.pts):
            if not u:
                continue
            pa, Ja = project(self.kind, x[t], a)
            pb, Jb = project(self.kind, x[t + d], b)
            r = pa - pb
            cost += (r ** 2).sum()
            blocks = [(t, Ja), (t + d, -Jb)]
            for f1, J1 in blocks:
                if f1 not in col:
                    continue
                i1 = col[f1] * P
                g[i1: i1 + P] += np.einsum("kri,kr->i", J1, r)
                for f2, J2 in blocks:
                    if f2 in col:
                        i2 = col[f2] * P
                        A[i1: i1 + P, i2: i2 + P] += np.einsum("kri,krj->ij", J1, J2)
        return cost, A, g

    def chain(self, x):
        """G_k; a disconnected frame sits at the pose of its nearest connected predecessor."""
        Ni = np.linalg.inv(self.N)
        eff = [max(q for q in range(k + 1) if self.conn[q]) for k in range(self.n)]
        return np.array([Ni @ matrix(self.kind, x[eff[k]]) @ self.N for k in range(self.n)])


def restatement(win, iterations):
    """The device's LM schedule: at most `iterations` builds, lambda0 = 1e-3 max diag, /10 on acceptance, *10 on a
    rejection or a failed factorisation, stop on a relative gain < 1e-12 or lambda > 1e16.  Returns (x, cost0, cost,
    accepted) with costs in normalised units."""
    x = win.x0.copy()
    cost, A, g = win.system(x)
    cost0, builds, accepted, done = cost, 1, 0, False
    dg = np.diag(A)
    lam = 1e-3 * dg.max() if len(dg) and dg.max() > 0 else 1e-3
    while builds < iterations and not done:
        delta = None
        while delta is None:
            try:
                Lc = np.linalg.cholesky(A + lam * np.eye(len(A)))
                delta = np.linalg.solve(Lc.T, np.linalg.solve(Lc, -g))
            except np.linalg.LinAlgError:
                lam *= 10.0
                if lam > 1e16:
                    done = True
                    break
        if done:
            break
        xt = x.copy()
        for i, k in enumerate(win.free):
            xt[k] = x[k] + delta[i * win.P: (i + 1) * win.P]
        ct, At, gt = win.system(xt)
        builds += 1
        if ct < cost:
            done = cost - ct < 1e-12 * cost
            x, cost, A, g = xt, ct, At, gt
            lam *= 0.1
            accepted += 1
        else:
            lam *= 10.0
            done = lam > 1e16
    return x, cost0, cost, accepted


def corner_dev(Ga, Gb, w, h):
    """max over frames and corners of |Ga_k c - Gb_k c| (px)."""
    c = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float64)
    return max(np.abs(map_pts(a, c) - map_pts(b, c)).max() for a, b in zip(Ga, Gb))


# ---- synthetic windows ----------------------------------------------------------------------------------------------
from niftymatch_b200.synth import camera_chain as true_chain, map_points as map_pts, span_window as window_arrays  # noqa: E402


def exact_window(kind, n, span, w, h, seed):
    """Noise-free float64 correspondences, all in the masks, and link models perturbed away from the truth."""
    rng = np.random.default_rng(seed)
    G, arrs = window_arrays(kind, n, span, w, h, 60, seed, noise=0.0, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.empty((L, 9))
    for l, (t, d) in enumerate(links(n, span)):
        M = np.linalg.inv(G[t + d]) @ G[t]
        M = M / M[2, 2]
        jit = np.zeros((3, 3))
        jit[:2, 2] = rng.normal(0, 2.0, 2)
        if kind >= 1:
            jit[:2, :2] = rng.normal(0, 2e-3, (2, 2)) * ([[1, 1], [1, 1]] if kind == 2 else 0)
        H[l] = (M + jit).reshape(-1)
    status = np.tile([1, 60, 0], (L, 1))
    masks = np.ones((L, 60), bool)
    return G, arrs, masks, H, status


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_restatement_recovers_exact_chains(kind):
    w, h, n, span = 640, 480, 8, 3
    G, arrs, masks, H, status = exact_window(kind, n, span, w, h, 40 + kind)
    win = Window(kind, n, span, w, h, *arrs, None, masks, H, status)
    assert corner_dev(win.chain(win.x0), G, w, h) > 1.0           # the perturbed links start the chain off the truth
    x, c0, c1, acc = restatement(win, 50)
    err = corner_dev(win.chain(x), G, w, h)
    assert err < 1e-9, (kind, err, c0, c1, acc)
    assert c1 <= c0 and acc >= 1


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_restatement_reaches_the_least_squares_minimum(kind):
    from scipy.optimize import least_squares
    w, h, n, span = 640, 480, 7, 2
    G, arrs = window_arrays(kind, n, span, w, h, 80, 50 + kind, noise=0.5, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.array([(np.linalg.inv(G[t + d]) @ G[t]).reshape(-1) for t, d in links(n, span)])
    win = Window(kind, n, span, w, h, *arrs, None, np.ones((L, 80), bool), H, np.tile([1, 80, 0], (L, 1)))
    x, _, _, _ = restatement(win, 100)
    P = NPAR[kind]

    def fun(v):
        xx = win.x0.copy()
        xx[1:] = v.reshape(n - 1, P)
        return win.residuals(xx).reshape(-1) / win.s           # pixels

    ls = least_squares(fun, win.x0[1:].reshape(-1), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=20000)
    xs = win.x0.copy()
    xs[1:] = ls.x.reshape(n - 1, P)
    err = corner_dev(win.chain(x), win.chain(xs), w, h)
    assert err < 1e-6, (kind, err)


# ---- on the device --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _frame_set(n, cap, seed):
    from niftymatch_b200 import synth
    rng = np.random.default_rng(seed)
    counts = [int(c) for c in rng.integers(300, cap, n)]
    counts[3], counts[5] = 0, cap                                    # an empty frame, a frame at capacity
    desc = (rng.random((n, cap, 128)) * 300).astype(np.float32)
    x = rng.uniform(0, 640, (n, cap)).astype(np.float32)
    y = rng.uniform(0, 480, (n, cap)).astype(np.float32)
    prev = None
    for f, c in enumerate(counts):
        if c == 0:
            prev = None
            continue
        d = synth.descriptors(c, 300 + f, planted_from=prev) if prev is not None else synth.descriptors(c, 300 + f)
        desc[f, :c] = d
        prev = d
    return desc, x, y, counts


@pytest.mark.gpu
def test_span_matching_and_alignment_equal_the_per_pair_calls(nm):
    """match_pairs_span at span 1 is bitwise match_pairs; every link (t, d) is bitwise nm_match_f32 (indices) and
    match_top2 (records) on its two frames, and align_pairs_span is bitwise align_points per link."""
    cap, n, span = 2048, 9, 3
    desc, x, y, counts = _frame_set(n, cap, 7)
    dd, xx, yy, cc = _cu(desc), _cu(x), _cu(y), torch.tensor(counts, dtype=torch.int32, device="cuda")
    init = torch.full((n_links(n, span), cap), 55, dtype=torch.int32, device="cuda")
    m1 = nm.match_pairs(dd, cc, 0.8, match_out=init[: n - 1].clone())
    s1 = nm.match_pairs_span(dd, cc, 1, 0.8, match_out=init[: n - 1].clone())
    assert torch.equal(m1, s1)
    m, rec, fb = nm.match_pairs_span(dd, cc, span, 0.8, match_out=init.clone(), want_records=True)
    corr = nm.align_pairs_span(xx, yy, m, cc, span)
    torch.cuda.synchronize()
    assert torch.equal(m[: n - 1], m1)
    mh, rh = m.cpu().numpy(), rec.cpu().numpy()
    nm.set_engine(0)
    try:
        for l, (t, d) in enumerate(links(n, span)):
            nA, nB = counts[t], counts[t + d]
            assert (mh[l, nA:] == 55).all(), (t, d)
            if nA == 0 or nB == 0:
                assert (mh[l] == 55).all(), (t, d)
            else:
                ref = nm.match(dd[t, :nA], dd[t + d, :nB], 0.8, match_io=init[l, :nA].clone()).cpu().numpy()
                r2 = nm.match_top2(dd[t, :nA], dd[t + d, :nB]).cpu().numpy()
                assert np.array_equal(mh[l, :nA], ref), (t, d)
                assert np.array_equal(rh[l, :nA].view(np.uint32)[:, :3], r2.view(np.uint32)[:, :3]), (t, d)
            mi = m[l].clone()
            mi[nA:] = -1
            mi[(mi >= nB) | (mi < 0)] = -1
            al = nm.align_points(xx[t], yy[t], xx[t + d], yy[t + d], mi.contiguous())
            for a, b in zip(corr, al):
                assert torch.equal(a[l], b), (t, d)
    finally:
        nm.set_engine(-1)
    assert (mh[link_row(n, 0, 2), : counts[0]] >= 0).sum() > 100     # planted chains survive a skip of two frames
    lib = nm.load()
    p = lambda t: C.c_void_p(t.data_ptr())
    for sp, nf in ((0, n), (9, n), (n, n), (2, 2)):
        assert lib.nm_match_pairs_span_f32(p(dd), p(cc), nf, cap, sp, 0.8, p(init), None, None, _stream()) == -1, (sp, nf)
        assert lib.nm_align_pairs_span_f32(p(xx), p(yy), p(init), p(cc), nf, cap, sp, *[p(c) for c in corr], _stream()) == -1


def device_window(nm, kind, n, span, w, h, seed, npts=2000, thr=4.0, rounds=0, iters=512):
    """window_arrays through ransac_batch per d (link seeds as StreamRegistrar) and refine_batch."""
    G, arrs = window_arrays(kind, n, span, w, h, npts, seed)
    d_ = [_cu(a) for a in arrs]
    HL, SL = [], []
    for d in range(1, span + 1):
        r0 = link_row(n, 0, d)
        Hd, Sd = nm.ransac_batch(kind, *[a[r0: r0 + n - d] for a in d_], None, thr, iters, seed + ((d - 1) << 40))
        HL.append(Hd)
        SL.append(Sd)
    HL, SL, mask = nm.refine_batch(kind, *d_, None, torch.cat(HL), torch.cat(SL), thr, rounds)
    return G, arrs, d_, HL, SL, mask


def placed_chain(nm, H, st, w, h):
    return nm.place(H, st, w, h).chain.cpu().numpy().reshape(-1, 3, 3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_adjustment_matches_the_restatement(nm, kind):
    """64-frame synthetic windows, 2 000 correspondences per link, sigma 0.3 px, 30 % outliers, span 3: chain_out matches
    the restatement on the same masks and link models within 1e-3 px at every frame corner, the chain place() rebuilds
    from H_out within 0.02 px, and the cost never rises."""
    w, h, n, span, thr = 640, 480, 64, 3, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 70 + kind)
    H, st, chain, rep = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, iterations=10)
    H, st, chain, rep = H.cpu().numpy(), st.cpu().numpy(), chain.cpu().numpy().reshape(n, 3, 3), rep.cpu().numpy()
    win = Window(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    x, c0, c1, acc = restatement(win, 10)
    ref = win.chain(x)
    err = corner_dev(chain, ref, w, h)
    placed = placed_chain(nm, torch.from_numpy(H).cuda(), torch.from_numpy(st).cuda(), w, h)
    perr = corner_dev(placed, ref, w, h)
    pts = sum(len(a) for (a, _), u in zip(win.pts, win.used) if u)
    print(f"kind {kind}: device vs restatement {err:.2e} px, placed chain {perr:.2e} px, mean squared residual "
          f"{rep[0]:.4f} -> {rep[1]:.4f} px^2 (restatement {c0 / win.s ** 2 / pts:.4f} -> {c1 / win.s ** 2 / pts:.4f}), "
          f"steps accepted {st[0, 2]} / {acc}")
    assert err < 1e-3 and perr < 0.02, (err, perr)
    assert rep[1] <= rep[0] and rep[2] == pts and rep[3] == sum(win.used)
    assert np.allclose(rep[:2], [c0 / win.s ** 2 / pts, c1 / win.s ** 2 / pts], rtol=1e-6)
    assert (st[:, 0] == 1).all()
    # status[:, 1]: the RANSAC rule on link (p, 1) with the adjusted model
    for p in (0, 31, 62):
        Hp = H[p].astype(np.float32)
        with np.errstate(all="ignore"):
            sx, sy, dx, dy = (a[p] for a in arrs)
            xq = Hp[0] * sx + Hp[1] * sy + Hp[2]
            yq = Hp[3] * sx + Hp[4] * sy + Hp[5]
            zq = Hp[6] * sx + Hp[7] * sy + Hp[8]
            d2 = (dx - xq / zq) ** 2 + (dy - yq / zq) ** 2
        assert abs(int(((sx >= 0) & (d2 < thr)).sum()) - st[p, 1]) <= 2, p


DRIFT_SCALE_BIAS = ("the mosaic-pixel cost is weighted by the local scale of G and on 64-frame windows rewards shrinking the "
                    "frames far from frame 0 (DESIGN 4.4.1): on an NVIDIA B200 the ratio was 0.73 for the similarity and "
                    "13.4 for the homography model")


def drift_ratio(nm, kind, windows=4, n=64, w=640, h=480, thr=4.0):
    """Mean over `windows` synthetic windows of the last frame's mean corner error: chained span-1 refits, span 3."""
    c = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float64)
    e1, e3 = [], []
    for wnd in range(windows):
        G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, 3, w, h, 90 + 10 * wnd + kind, rounds=2)
        last = lambda Gk: np.hypot(*(map_pts(Gk[-1], c) - map_pts(G[-1], c)).T).mean()
        e1.append(last(placed_chain(nm, HL[: n - 1].contiguous(), SL[: n - 1].contiguous(), w, h)))
        _, _, chain, _ = nm.adjust_chain(kind, *d_, None, 3, mask, HL, SL, w, h, thr)
        e3.append(last(chain.cpu().numpy().reshape(n, 3, 3)))
    return float(np.mean(e1)), float(np.mean(e3))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, pytest.param(1, marks=pytest.mark.xfail(strict=True, reason=DRIFT_SCALE_BIAS)),
                                  pytest.param(2, marks=pytest.mark.xfail(strict=True, reason=DRIFT_SCALE_BIAS))])
def test_span_three_halves_the_drift_of_chained_refits(nm, kind):
    """The synthetic 64-frame windows (2 000 correspondences per link, sigma 0.3 px, 30 % outliers), four per kind: span 3
    must bring the last frame's mean corner error to at most half that of the chained span-1 refits (a resistor-network
    estimate for equal-noise links predicts about 1/sqrt(14)).  The translation model meets the bound (0.08); the
    similarity model lowers the drift without halving it and the homography model raises it (strict xfail, ratios
    printed) -- see DRIFT_SCALE_BIAS."""
    e1, e3 = drift_ratio(nm, kind)
    print(f"kind {kind}: last frame mean corner error over 4 windows, chained span-1 refits {e1:.4f} px, span 3 "
          f"{e3:.4f} px, ratio {e3 / e1:.3f}")
    assert e3 <= 0.5 * e1, (e1, e3, e3 / e1)


@pytest.mark.gpu
def test_skip_links_bridge_a_failed_pair(nm):
    """Consecutive link 20 loses its model: the span-2 link (19, 21) bridges it, status_out marks the pair connected and
    place() rebuilds the restatement's chain.  A frame without any usable link is flagged disconnected and sits at its
    predecessor's pose; the pair after it reproduces the next frame's pose."""
    kind, w, h, n, span, thr = 2, 640, 480, 32, 2, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 120, npts=1000)
    SL = SL.clone()
    SL[20, 0] = 0                                                     # pair (20, 21)
    for t, d in ((9, 1), (8, 2)):                                     # no usable link reaches frame 10; (9, 2) bridges it
        SL[link_row(n, t, d), 0] = 0
    H, st, chain, _ = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr)
    win = Window(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    assert win.conn[21] and not win.conn[10] and sum(win.conn) == n - 1
    x, _, _, _ = restatement(win, 10)
    ref = win.chain(x)
    st_h, chain = st.cpu().numpy(), chain.cpu().numpy().reshape(n, 3, 3)
    assert st_h[20, 0] == 1 and st_h[9].tolist() == [0, 0, 0] and (np.delete(st_h[:, 0], 9) == 1).all()
    assert np.array_equal(H[9].cpu().numpy().view(np.int32), HL[9].cpu().numpy().view(np.int32))
    assert np.array_equal(chain[10], chain[9])
    placed = placed_chain(nm, H, st, w, h)
    assert corner_dev(chain, ref, w, h) < 1e-3
    assert corner_dev(placed, ref, w, h) < 0.02


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 2])
def test_adjustment_is_reproducible_in_place_and_graph_capturable(nm, kind):
    w, h, n, span, thr = 640, 480, 24, 3, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 140 + kind, npts=800)
    counts = torch.full((n_links(n, span),), 800, dtype=torch.int32, device="cuda")
    out = nm.adjust_chain(kind, *d_, counts, span, mask, HL, SL, w, h, thr)
    again = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr)
    for a, b in zip(out, again):
        assert torch.equal(a, b)
    Hi, Si = HL.clone(), SL.clone()
    res = nm.adjust_chain(kind, *d_, None, span, mask, Hi, Si, w, h, thr, out=(Hi[: n - 1], Si[: n - 1]))
    assert torch.equal(res[0], out[0]) and torch.equal(res[1], out[1]) and torch.equal(res[2], out[2])
    assert torch.equal(Hi[: n - 1], out[0]) and torch.equal(Hi[n - 1:], HL[n - 1:])
    Hg, Sg = torch.empty_like(out[0]), torch.empty_like(out[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg))
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    Hg.zero_()
    Sg.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, _, cg, rg = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg))
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(Hg, out[0]) and torch.equal(Sg, out[1]) and torch.equal(cg, out[2]) and torch.equal(rg, out[3])
    # argument checks
    lib = nm.load()
    p = lambda t: C.c_void_p(t.data_ptr())
    Ho, So = torch.empty(n - 1, 9, device="cuda"), torch.empty(n - 1, 3, dtype=torch.int32, device="cuda")

    def call(kind=kind, n_frames=n, span=span, sx=p(d_[0]), masks=p(mask), Hl=p(HL), Sl=p(SL), Hout=p(Ho), Sout=p(So), it=10):
        return lib.nm_ransac_adjust_chain_f32(kind, sx, p(d_[1]), p(d_[2]), p(d_[3]), 800, None, 800, thr, n_frames, span, w, h,
                                              masks, Hl, Sl, it, Hout, Sout, None, None, _stream())
    assert call() == 0
    for bad in (dict(kind=3), dict(kind=-1), dict(span=0), dict(span=9), dict(n_frames=3, span=3), dict(n_frames=1025),
                dict(sx=None), dict(masks=None), dict(Hl=None), dict(Sl=None), dict(Hout=None), dict(Sout=None), dict(it=0)):
        assert call(**bad) == -1, bad
    torch.cuda.synchronize()


# ---- the stream pipeline ---------------------------------------------------------------------------------------------
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


def _stream_errors(nm, H, st, w, h, offs):
    n = len(offs)
    G = placed_chain(nm, H, st, w, h)
    c1 = np.array([[0, 0, 1.0], [w - 1, 0, 1], [0, h - 1, 1], [w - 1, h - 1, 1]]).T
    true = np.array([(ox - offs[0][0], oy - offs[0][1]) for ox, oy in offs], np.float64)
    return max(np.abs((G[k] @ c1)[:2] / (G[k] @ c1)[2] - c1[:2] - true[k][:, None]).max() for k in range(n))


@pytest.mark.gpu
def test_sift_crop_stream_with_span_three(nm):
    """The 24-frame SIFT crop stream of test_refined_homography_stream_drifts_less: with the homography model (threshold
    0.5 px, two refit rounds) span 3 lowers the chained corner error below the span-1 one; the translation model keeps
    its < 1 px."""
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n, offs, bgra = _crop_stream()
    fr = torch.from_numpy(bgra).cuda()
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 8, 8192)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    errs = {}
    for span in (1, 3):
        reg = StreamRegistrar(sb, chunk=8, kind=nm.HOMOGRAPHY, inlier_threshold=0.25, iterations=512, seed=3, refine_rounds=2,
                              span=span)
        H, st = reg.run(frames_of, 0, n)
        assert (st[:, 0] == 1).all()
        errs[span] = _stream_errors(nm, H, st, w, h, offs)
    reg = StreamRegistrar(sb, chunk=8, kind=nm.TRANSLATION, inlier_threshold=0.25, iterations=512, seed=3, refine_rounds=2, span=3)
    H, st = reg.run(frames_of, 0, n)
    e_t = _stream_errors(nm, H, st, w, h, offs)
    sb.close()
    print(f"homography crop stream, worst corner error: span 1 {errs[1]:.3f} px, span 3 {errs[3]:.3f} px; "
          f"translation span 3 {e_t:.3f} px")
    assert errs[3] < errs[1], errs
    assert e_t < 1.0, e_t


@pytest.mark.gpu
def test_stream_registrar_span_equals_the_public_calls(nm):
    """StreamRegistrar(span=3) equals, bitwise, the five public calls composed by hand per window (chunk 5 over 11
    frames, so the last window is shorter than span + 1 and uses span 2); StreamRegistrar(span=1) equals the default."""
    from niftymatch_b200 import synth
    from niftymatch_b200.dist import StreamRegistrar
    w, h = 512, 384
    base = synth.scene(w + 80, h + 80, synth.SEED_BASE + 9)
    offs = [(8 + 6 * k, 8 + 5 * k - (k % 3)) for k in range(11)]
    fr = _cu(np.stack([base[oy: oy + h, ox: ox + w] for ox, oy in offs]))
    n = len(offs)
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 5, 8192)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    kw = dict(kind=nm.HOMOGRAPHY, inlier_threshold=1.0, iterations=512, seed=5, refine_rounds=1)
    H0, s0 = StreamRegistrar(sb, chunk=5, **kw).run(frames_of, 0, n)
    H1, s1 = StreamRegistrar(sb, chunk=5, span=1, **kw).run(frames_of, 0, n)
    assert torch.equal(H0, H1) and torch.equal(s0, s1)
    H3, s3 = StreamRegistrar(sb, chunk=5, span=3, **kw).run(frames_of, 0, n)
    Hr, sr = torch.zeros_like(H3), torch.zeros_like(s3)
    c0 = 0
    while c0 < n - 1:
        c1 = min(n, c0 + 5)
        m = c1 - c0
        S = min(3, m - 1)
        sb.run(frames_of(c0, c1))
        r = sb.results()
        cnt = r["counts"][:m]
        mt = nm.match_pairs_span(r["desc"][:m], cnt, S, 0.8)
        corr = nm.align_pairs_span(r["x"][:m], r["y"][:m], mt, cnt, S)
        HL, SL = [], []
        for d in range(1, S + 1):
            r0 = link_row(m, 0, d)
            a, b = nm.ransac_batch(nm.HOMOGRAPHY, *[c[r0: r0 + m - d] for c in corr], cnt[: m - d], 1.0, 512, 5 + c0 + ((d - 1) << 40))
            HL.append(a)
            SL.append(b)
        lc = torch.cat([cnt[: m - d] for d in range(1, S + 1)])
        HL, SL, mk = nm.refine_batch(nm.HOMOGRAPHY, *corr, lc, torch.cat(HL), torch.cat(SL), 1.0, 1)
        Ha, Sa, _, _ = nm.adjust_chain(nm.HOMOGRAPHY, *corr, lc, S, mk, HL, SL, w, h, 1.0, 10)
        Hr[c0: c1 - 1], sr[c0: c1 - 1] = Ha, Sa
        c0 = c1 - 1
    sb.close()
    assert torch.equal(H3, Hr) and torch.equal(s3, sr)
    assert (s3[:, 0] == 1).all()
