"""The transfer cost of the chain adjustment (nm_ransac_adjust_chain_cost_f32 with NM_ADJUST_TRANSFER,
adjust_chain(cost=TRANSFER), StreamRegistrar(adjust_cost=TRANSFER)).

Each link's residual is pi(G_(t+d)^-1 G_t s_i) - d_i in the pixels of its target frame, so it depends on the relative
poses only.  A float64 restatement (the mosaic-cost restatement of test_gpu_chain_adjust with this residual and its
Jacobians) is checked without a GPU: it recovers exact chains, reaches scipy.optimize.least_squares' minimum and, for
the translation model, equals the mosaic cost.  The GPU tests compare the device with it, measure drift, and check
that cost 0 through the new entry is bitwise the existing entry."""
import ctypes as C
import hashlib

import numpy as np
import pytest
import torch

from tests.test_gpu_chain_adjust import (NPAR, Window, restatement, links, link_row, n_links, matrix, corner_dev, exact_window,
                                         window_arrays, map_pts, device_window, placed_chain, _cu, _stream, _crop_stream,
                                         _stream_errors)

MOSAIC, TRANSFER = 0, 1


# ---- the restatement ------------------------------------------------------------------------------------------------
def _dmat(kind, v):
    """d(Gn(th) v) / d th for homogeneous points v (k, 3): (k, 3, P)."""
    k = len(v)
    D = np.zeros((k, 3, NPAR[kind]))
    if kind == 0:
        D[:, 0, 0] = D[:, 1, 1] = v[:, 2]
    elif kind == 1:
        D[:, 0, 0], D[:, 1, 0] = v[:, 0], v[:, 1]
        D[:, 0, 1], D[:, 1, 1] = -v[:, 1], v[:, 0]
        D[:, 0, 2] = D[:, 1, 3] = v[:, 2]
    else:
        for i in range(8):
            D[:, i // 3, i] = v[:, i % 3]
    return D


class TransferWindow(Window):
    """Window with the transfer residual pi(Gn_u^-1 Gn_t a) - b, u = t + d (normalised units of frame u)."""

    def link(self, x, t, d, a, b):
        """(r (k, 2), dr/dth_t, dr/dth_u (k, 2, P), every p3 > 0 and r finite)"""
        Gi = np.linalg.inv(matrix(self.kind, x[t + d]))
        ah = np.c_[a, np.ones(len(a))]
        with np.errstate(all="ignore"):
            p = ah @ (Gi @ matrix(self.kind, x[t])).T
            iw = 1.0 / p[:, 2]
            U, V = p[:, 0] * iw, p[:, 1] * iw
            r = np.stack([U, V], 1) - b
            z, o = np.zeros(len(a)), np.ones(len(a))
            dpi = iw[:, None, None] * np.stack([np.stack([o, z, -U], 1), np.stack([z, o, -V], 1)], 1)
            A = dpi @ Gi
            Jt = A @ _dmat(self.kind, ah)
            Ju = -(A @ _dmat(self.kind, p))
        return r, Jt, Ju, bool((p[:, 2] > 0).all() and np.isfinite(r).all())

    def residuals(self, x):
        out = [self.link(x, t, d, a, b)[0] for (t, d), u, (a, b) in zip(self.order, self.used, self.pts) if u]
        return np.concatenate(out) if out else np.zeros((0, 2))

    def system(self, x):
        """cost (+inf when a point has p3 <= 0 or a non-finite residual), J^T J and J^T r over the free frames."""
        P, col = self.P, {k: i for i, k in enumerate(self.free)}
        A = np.zeros((len(self.free) * P,) * 2)
        g = np.zeros(len(self.free) * P)
        cost, finite = 0.0, True
        for (t, d), u, (a, b) in zip(self.order, self.used, self.pts):
            if not u:
                continue
            r, Jt, Ju, ok = self.link(x, t, d, a, b)
            finite = finite and ok
            cost += (r ** 2).sum()
            blocks = [(t, Jt), (t + d, Ju)]
            for f1, J1 in blocks:
                if f1 not in col:
                    continue
                i1 = col[f1] * P
                g[i1: i1 + P] += np.einsum("kri,kr->i", J1, r)
                for f2, J2 in blocks:
                    if f2 in col:
                        i2 = col[f2] * P
                        A[i1: i1 + P, i2: i2 + P] += np.einsum("kri,krj->ij", J1, J2)
        return (cost if finite else np.inf), A, g


def transfer_restatement(win, iterations):
    """The device's LM schedule on the transfer cost: a +inf cost at the initial point leaves the window as it is."""
    if not np.isfinite(win.system(win.x0)[0]):
        return win.x0.copy(), np.inf, np.inf, 0
    return restatement(win, iterations)


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_transfer_restatement_recovers_exact_chains(kind):
    w, h, n, span = 640, 480, 8, 3
    G, arrs, masks, H, status = exact_window(kind, n, span, w, h, 40 + kind)
    win = TransferWindow(kind, n, span, w, h, *arrs, None, masks, H, status)
    assert corner_dev(win.chain(win.x0), G, w, h) > 1.0
    x, c0, c1, acc = transfer_restatement(win, 50)
    err = corner_dev(win.chain(x), G, w, h)
    assert err < 1e-9, (kind, err, c0, c1, acc)
    assert c1 <= c0 and acc >= 1


@pytest.mark.parametrize("kind", [0, 1, 2])
def test_transfer_restatement_reaches_the_least_squares_minimum(kind):
    from scipy.optimize import least_squares
    w, h, n, span = 640, 480, 7, 2
    G, arrs = window_arrays(kind, n, span, w, h, 80, 50 + kind, noise=0.5, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.array([(np.linalg.inv(G[t + d]) @ G[t]).reshape(-1) for t, d in links(n, span)])
    win = TransferWindow(kind, n, span, w, h, *arrs, None, np.ones((L, 80), bool), H, np.tile([1, 80, 0], (L, 1)))
    x, _, _, _ = transfer_restatement(win, 100)
    P = NPAR[kind]

    def fun(v):
        xx = win.x0.copy()
        xx[1:] = v.reshape(n - 1, P)
        return win.residuals(xx).reshape(-1) / win.s

    ls = least_squares(fun, win.x0[1:].reshape(-1), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=20000)
    xs = win.x0.copy()
    xs[1:] = ls.x.reshape(n - 1, P)
    err = corner_dev(win.chain(x), win.chain(xs), w, h)
    assert err < 1e-6, (kind, err)


def test_transfer_restatement_equals_the_mosaic_cost_for_translation():
    """a + t_t - t_u - b is the residual of both costs for the translation model."""
    w, h, n, span = 640, 480, 12, 3
    G, arrs = window_arrays(0, n, span, w, h, 80, 61, noise=0.5, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.array([(np.linalg.inv(G[t + d]) @ G[t]).reshape(-1) + np.r_[0, 0, 1.5, 0, 0, -1.0, 0, 0, 0] for t, d in links(n, span)])
    args = (0, n, span, w, h, *arrs, None, np.ones((L, 80), bool), H, np.tile([1, 80, 0], (L, 1)))
    mw, tw = Window(*args), TransferWindow(*args)
    xm, m0, m1, _ = restatement(mw, 20)
    xt, t0, t1, _ = transfer_restatement(tw, 20)
    assert np.isclose(m0, t0, rtol=1e-12) and np.isclose(m1, t1, rtol=1e-9)
    err = corner_dev(mw.chain(xm), tw.chain(xt), w, h)
    assert err < 1e-9, err


# ---- on the device --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_transfer_adjustment_matches_the_restatement(nm, kind):
    """The 64-frame span-3 windows of test_adjustment_matches_the_restatement with the transfer cost: chain_out within
    1e-3 px of the restatement, the chain place() rebuilds from H_out within 0.02 px, the report equal to the
    restatement's costs, and the cost never rises."""
    w, h, n, span, thr = 640, 480, 64, 3, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 70 + kind)
    H, st, chain, rep = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, iterations=10, cost=nm.TRANSFER)
    H, st, chain, rep = H.cpu().numpy(), st.cpu().numpy(), chain.cpu().numpy().reshape(n, 3, 3), rep.cpu().numpy()
    win = TransferWindow(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    x, c0, c1, acc = transfer_restatement(win, 10)
    ref = win.chain(x)
    err = corner_dev(chain, ref, w, h)
    placed = placed_chain(nm, torch.from_numpy(H).cuda(), torch.from_numpy(st).cuda(), w, h)
    perr = corner_dev(placed, ref, w, h)
    pts = sum(len(a) for (a, _), u in zip(win.pts, win.used) if u)
    print(f"kind {kind}, transfer cost: device vs restatement {err:.2e} px, placed chain {perr:.2e} px, mean squared "
          f"residual {rep[0]:.4f} -> {rep[1]:.4f} px^2 (restatement {c0 / win.s ** 2 / pts:.4f} -> "
          f"{c1 / win.s ** 2 / pts:.4f}), steps accepted {st[0, 2]} / {acc}")
    assert err < 1e-3 and perr < 0.02, (err, perr)
    assert rep[1] <= rep[0] and rep[2] == pts and rep[3] == sum(win.used)
    assert np.allclose(rep[:2], [c0 / win.s ** 2 / pts, c1 / win.s ** 2 / pts], rtol=1e-6)
    assert (st[:, 0] == 1).all()


def drift(nm, kind, cost, windows=4, n=64, w=640, h=480, thr=4.0):
    """drift_ratio of test_gpu_chain_adjust (same windows and seeds) with a choice of cost: the mean over the windows of
    the last frame's mean corner error for chained span-1 refits and for the span-3 adjustment."""
    c = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float64)
    e1, e3 = [], []
    for wnd in range(windows):
        G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, 3, w, h, 90 + 10 * wnd + kind, rounds=2)
        last = lambda Gk: np.hypot(*(map_pts(Gk[-1], c) - map_pts(G[-1], c)).T).mean()
        e1.append(last(placed_chain(nm, HL[: n - 1].contiguous(), SL[: n - 1].contiguous(), w, h)))
        _, _, chain, _ = nm.adjust_chain(kind, *d_, None, 3, mask, HL, SL, w, h, thr, cost=cost)
        e3.append(last(chain.cpu().numpy().reshape(n, 3, 3)))
    return float(np.mean(e1)), float(np.mean(e3))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_transfer_span_three_halves_the_drift_of_chained_refits(nm, kind):
    """The bound of test_span_three_halves_the_drift_of_chained_refits (span 3 at most half the last frame's mean corner
    error of chained span-1 refits, four synthetic 64-frame windows) with the transfer cost, for every kind."""
    e1, e3 = drift(nm, kind, TRANSFER)
    print(f"kind {kind}, transfer cost: last frame mean corner error over 4 windows, chained span-1 refits {e1:.4f} px, "
          f"span 3 {e3:.4f} px, ratio {e3 / e1:.3f}")
    assert e3 <= 0.5 * e1, (e1, e3, e3 / e1)


@pytest.mark.gpu
def test_sift_crop_stream_with_the_transfer_cost(nm):
    """The 24-frame SIFT crop stream (homography, 0.5 px threshold, two refit rounds, 8-frame windows): with the
    transfer cost span 3 has a lower worst chained corner error than span 1."""
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n, offs, bgra = _crop_stream()
    fr = torch.from_numpy(bgra).cuda()
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 8, 8192)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    errs = {}
    for span, cost in ((1, MOSAIC), (3, MOSAIC), (3, TRANSFER)):
        reg = StreamRegistrar(sb, chunk=8, kind=nm.HOMOGRAPHY, inlier_threshold=0.25, iterations=512, seed=3, refine_rounds=2,
                              span=span, adjust_cost=cost)
        H, st = reg.run(frames_of, 0, n)
        assert (st[:, 0] == 1).all()
        errs[span, cost] = _stream_errors(nm, H, st, w, h, offs)
    sb.close()
    print(f"homography crop stream, worst corner error: span 1 {errs[1, MOSAIC]:.3f} px, span 3 mosaic cost "
          f"{errs[3, MOSAIC]:.3f} px, span 3 transfer cost {errs[3, TRANSFER]:.3f} px")
    assert errs[3, TRANSFER] < errs[1, MOSAIC], errs


# sha256 of H_out, status_out, chain_out and report_out of nm_ransac_adjust_chain_f32 on the windows of _digest_window,
# as the build before the transfer cost computed them (NVIDIA B200)
MOSAIC_DIGESTS = {0: "a78d6515868e7d99bcf87f1b76d461061a9bdc0def1edb69b1ef33d3dd11f78e",
                  1: "fcf5acd8ffbf5eac83ab0e72d8b1a4de7883d0ef7af98a29c55a1c992ab63ea9",
                  2: "b2d43eccadcb6696e57d1a22c494cc456d247fe09bd8f49086de8aaef3445361"}


def _digest_window(nm, kind):
    w, h, n, span = 640, 480, 24, 3
    return (w, h, n, span) + device_window(nm, kind, n, span, w, h, 160 + kind, npts=800)[2:]


def _entry(nm, name, *pre, kind, d_, span, mask, HL, SL, w, h, n, thr=4.0, it=10):
    p = lambda t: C.c_void_p(t.data_ptr())
    out = (torch.empty(n - 1, 9, device="cuda"), torch.empty(n - 1, 3, dtype=torch.int32, device="cuda"),
           torch.empty(n, 9, dtype=torch.float64, device="cuda"), torch.empty(4, dtype=torch.float64, device="cuda"))
    rc = getattr(nm.load(), name)(kind, *pre, *[p(a) for a in d_], d_[0].shape[1], None, d_[0].shape[1], thr, n, span, w, h,
                                  p(mask), p(HL), p(SL), it, *[p(o) for o in out], _stream())
    assert rc == 0, rc
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_mosaic_cost_through_the_new_entry_is_the_existing_entry(nm, kind):
    """Cost 0 of nm_ransac_adjust_chain_cost_f32 and adjust_chain's default are bitwise nm_ransac_adjust_chain_f32 (all
    four outputs), and those outputs are bitwise what the build before the transfer cost returned."""
    w, h, n, span, d_, HL, SL, mask = _digest_window(nm, kind)
    kw = dict(kind=kind, d_=d_, span=span, mask=mask, HL=HL, SL=SL, w=w, h=h, n=n)
    old = _entry(nm, "nm_ransac_adjust_chain_f32", **kw)
    new = _entry(nm, "nm_ransac_adjust_chain_cost_f32", MOSAIC, **kw)
    default = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, 4.0)
    for a, b, c in zip(old, new, default):
        assert torch.equal(a, b) and torch.equal(a, c)
    digest = hashlib.sha256(b"".join(t.cpu().numpy().tobytes() for t in old)).hexdigest()
    print(f"kind {kind}: mosaic-cost digest {digest}")
    assert digest == MOSAIC_DIGESTS[kind], digest


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 2])
def test_transfer_adjustment_is_reproducible_in_place_and_graph_capturable(nm, kind):
    w, h, n, span, thr = 640, 480, 24, 3, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 140 + kind, npts=800)
    T = nm.TRANSFER
    counts = torch.full((n_links(n, span),), 800, dtype=torch.int32, device="cuda")
    out = nm.adjust_chain(kind, *d_, counts, span, mask, HL, SL, w, h, thr, cost=T)
    again = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=T)
    for a, b in zip(out, again):
        assert torch.equal(a, b)
    assert out[1][0, 2].item() >= 1
    Hi, Si = HL.clone(), SL.clone()
    res = nm.adjust_chain(kind, *d_, None, span, mask, Hi, Si, w, h, thr, out=(Hi[: n - 1], Si[: n - 1]), cost=T)
    assert torch.equal(res[0], out[0]) and torch.equal(res[1], out[1]) and torch.equal(res[2], out[2])
    assert torch.equal(Hi[: n - 1], out[0]) and torch.equal(Hi[n - 1:], HL[n - 1:])
    Hg, Sg = torch.empty_like(out[0]), torch.empty_like(out[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg), cost=T)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    Hg.zero_()
    Sg.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, _, cg, rg = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg), cost=T)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(Hg, out[0]) and torch.equal(Sg, out[1]) and torch.equal(cg, out[2]) and torch.equal(rg, out[3])
    # argument checks
    lib = nm.load()
    p = lambda t: C.c_void_p(t.data_ptr())
    Ho, So = torch.empty(n - 1, 9, device="cuda"), torch.empty(n - 1, 3, dtype=torch.int32, device="cuda")

    def call(kind=kind, cost=T, n_frames=n, span=span, sx=p(d_[0]), masks=p(mask), Hl=p(HL), Sl=p(SL), Hout=p(Ho), Sout=p(So),
             it=10):
        return lib.nm_ransac_adjust_chain_cost_f32(kind, cost, sx, p(d_[1]), p(d_[2]), p(d_[3]), 800, None, 800, thr, n_frames,
                                                   span, w, h, masks, Hl, Sl, it, Hout, Sout, None, None, _stream())
    assert call() == 0 and call(cost=MOSAIC) == 0
    for bad in (dict(cost=2), dict(cost=-1), dict(kind=3), dict(kind=-1), dict(span=0), dict(span=9), dict(n_frames=3, span=3),
                dict(n_frames=1025), dict(sx=None), dict(masks=None), dict(Hl=None), dict(Sl=None), dict(Hout=None),
                dict(Sout=None), dict(it=0)):
        assert call(**bad) == -1, bad
    with pytest.raises(nm.NmError):
        nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=2)
    torch.cuda.synchronize()


@pytest.mark.gpu
def test_transfer_skip_links_bridge_a_failed_pair(nm):
    """test_skip_links_bridge_a_failed_pair with the transfer cost: consecutive link 20 bridged by (19, 21), frame 10
    disconnected and at its predecessor's pose, chain and placed chain on the transfer restatement's."""
    kind, w, h, n, span, thr = 2, 640, 480, 32, 2, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 120, npts=1000)
    SL = SL.clone()
    SL[20, 0] = 0
    for t, d in ((9, 1), (8, 2)):
        SL[link_row(n, t, d), 0] = 0
    H, st, chain, _ = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=nm.TRANSFER)
    win = TransferWindow(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    assert win.conn[21] and not win.conn[10] and sum(win.conn) == n - 1
    x, _, _, _ = transfer_restatement(win, 10)
    ref = win.chain(x)
    st_h, chain = st.cpu().numpy(), chain.cpu().numpy().reshape(n, 3, 3)
    assert st_h[20, 0] == 1 and st_h[9].tolist() == [0, 0, 0] and (np.delete(st_h[:, 0], 9) == 1).all()
    assert np.array_equal(H[9].cpu().numpy().view(np.int32), HL[9].cpu().numpy().view(np.int32))
    assert np.array_equal(chain[10], chain[9])
    placed = placed_chain(nm, H, st, w, h)
    assert corner_dev(chain, ref, w, h) < 1e-3
    assert corner_dev(placed, ref, w, h) < 0.02


@pytest.mark.gpu
def test_a_point_behind_the_camera_leaves_the_window_unadjusted(nm):
    """One mask point of link (0, 1) placed where the initial Gn_1^-1 Gn_0 gives it p3 = -1: the transfer cost is +inf at
    the initial poses, so the window keeps its initial chain (bitwise the one-build result), with 0 LM steps and +inf
    costs in the report.  Without that point the same window is adjusted."""
    kind, w, h, n, span, thr = 2, 640, 480, 16, 2, 4.0
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 150, npts=600)
    free = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=nm.TRANSFER)
    assert free[1][0, 2].item() >= 1 and np.isfinite(free[3].cpu().numpy()[:2]).all()
    win = TransferWindow(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    M = np.linalg.inv(matrix(kind, win.x0[1])) @ matrix(kind, win.x0[0])
    an = -(1.0 + M[2, 2]) * M[2, :2] / (M[2, :2] ** 2).sum()      # M[2] . (an, 1) = -1
    px = an / win.s + [0.5 * (w - 1), 0.5 * (h - 1)]
    arrs = [a.copy() for a in arrs]
    arrs[0][0, 0], arrs[1][0, 0] = px
    d_ = [_cu(a) for a in arrs]
    mask = mask.clone()
    mask[0, 0] = True
    win = TransferWindow(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy())
    assert win.link(win.x0, 0, 1, *win.pts[0])[3] is False
    x, c0, c1, acc = transfer_restatement(win, 10)
    assert acc == 0 and np.isinf(c0) and np.isinf(c1)
    H, st, chain, rep = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=nm.TRANSFER)
    H1, st1, chain1, _ = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, iterations=1)
    assert torch.equal(H, H1) and torch.equal(st, st1) and torch.equal(chain, chain1)
    assert (st[:, 2] == 0).all() and (st[:, 0] == 1).all()
    rep = rep.cpu().numpy()
    assert np.isinf(rep[0]) and np.isinf(rep[1]) and rep[3] == sum(win.used)
    assert corner_dev(chain.cpu().numpy().reshape(n, 3, 3), win.chain(x), w, h) < 1e-6


@pytest.mark.gpu
def test_stream_registrar_transfer_cost_equals_the_public_calls(nm):
    """StreamRegistrar(span=3, adjust_cost=TRANSFER) equals, bitwise, the public calls composed by hand per window
    (chunk 5 over 11 frames, the last window at span 2)."""
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
    H3, s3 = StreamRegistrar(sb, chunk=5, span=3, adjust_cost=nm.TRANSFER, **kw).run(frames_of, 0, n)
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
        Ha, Sa, _, _ = nm.adjust_chain(nm.HOMOGRAPHY, *corr, lc, S, mk, HL, SL, w, h, 1.0, 10, cost=nm.TRANSFER)
        Hr[c0: c1 - 1], sr[c0: c1 - 1] = Ha, Sa
        c0 = c1 - 1
    sb.close()
    assert torch.equal(H3, Hr) and torch.equal(s3, sr)
    assert (s3[:, 0] == 1).all()
