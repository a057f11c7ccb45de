"""Chain adjustment with fixed frames (nm_ransac_adjust_chain_fixed_f32, adjust_chain(fixed=...),
StreamRegistrar(overlap=O), StreamRegistrar.run(resume=True)).

Frames 0 .. n_fixed-1 of a window keep given poses (rebased on the first of them) and only links that reach a later
frame are used, so consecutive windows that share `overlap` frames use every skip link that crosses their boundary.
The float64 restatements of test_gpu_chain_adjust and test_gpu_chain_adjust_transfer, with the fixed frames taken out
of the unknowns, are checked without a GPU; the GPU tests compare the device with them, pin n_fixed = 1 to the
existing entry, and measure what the overlap does to drift."""
import ctypes as C
import hashlib

import numpy as np
import pytest
import torch

from tests.test_gpu_chain_adjust import (MINPTS, NPAR, Window, restatement, links, link_row, n_links, params, corner_dev,
                                         exact_window, window_arrays, map_pts, device_window, placed_chain, _chain_step,
                                         _renormalise, _cu, _stream, _crop_stream, _stream_errors)
from tests.test_gpu_chain_adjust_transfer import (TransferWindow, transfer_restatement, MOSAIC_DIGESTS, _digest_window,
                                                  MOSAIC, TRANSFER)


# ---- the restatement ------------------------------------------------------------------------------------------------
class Fixed:
    """Frames 0 .. nf-1 held at F (nf, 3, 3), frame j -> frame-0 pixels (F[0] = I); fconn[j] false, or a non-finite
    F[j], makes fixed frame j disconnected (pose of its predecessor).  Free frames k >= nf take the usual initial pose
    rule (frame k - d may be fixed), a link is used only if its later frame is free, and the unknowns are the connected
    free frames."""

    def __init__(self, kind, n, span, w, h, sx, sy, dx, dy, counts, masks, H, status, F, fconn=None):
        super().__init__(kind, n, span, w, h, sx, sy, dx, dy, counts, masks, H, status)
        nf, L = len(F), n_links(n, span)
        H = np.asarray(H).reshape(L, 9)
        status = np.asarray(status).reshape(L, 3)
        usable = [status[l, 0] == 1 and len(self.pts[l][0]) >= MINPTS[kind] for l in range(L)]
        G, self.conn = [np.eye(3)], [True]
        for j in range(1, nf):
            ok = (fconn is None or bool(fconn[j])) and bool(np.isfinite(F[j]).all())
            G.append(np.asarray(F[j], np.float64) if ok else G[j - 1].copy())
            self.conn.append(ok)
        for k in range(nf, n):
            for d in range(1, min(span, k) + 1):
                l = link_row(n, k - d, d)
                if self.conn[k - d] and usable[l]:
                    G.append(_renormalise(G[k - d] @ _chain_step(H[l])))
                    self.conn.append(True)
                    break
            else:
                G.append(G[k - 1].copy())
                self.conn.append(False)
        self.nf = nf
        self.x0 = np.array([params(kind, self.N @ g @ np.linalg.inv(self.N)) for g in G])
        self.x0[0] = params(kind, np.eye(3))
        self.used = [usable[link_row(n, t, d)] and t + d >= nf and self.conn[t] and self.conn[t + d] for t, d in links(n, span)]
        self.free = [k for k in range(nf, n) if self.conn[k]]


class FixedWindow(Fixed, Window):
    pass


class FixedTransferWindow(Fixed, TransferWindow):
    pass


WINDOWS = {MOSAIC: (FixedWindow, restatement), TRANSFER: (FixedTransferWindow, transfer_restatement)}


def shifted(F, px, seed):
    """F_j moved by a translation of about `px` pixels (j >= 1): fixed poses that disagree with the links."""
    rng = np.random.default_rng(seed)
    out = [np.eye(3)]
    for f in F[1:]:
        T = np.eye(3)
        T[:2, 2] = rng.normal(0, px, 2)
        out.append(T @ f)
    return np.array(out)


@pytest.mark.parametrize("cost", [MOSAIC, TRANSFER])
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_fixed_restatement_recovers_exact_chains(kind, cost):
    """Fixed frames at the true poses, the free frames started off the truth by perturbed links: exact chains."""
    w, h, n, span, nf = 640, 480, 8, 3, 3
    Wc, solve = WINDOWS[cost]
    G, arrs, masks, H, status = exact_window(kind, n, span, w, h, 40 + kind)
    win = Wc(kind, n, span, w, h, *arrs, None, masks, H, status, F=G[:nf])
    assert win.free == list(range(nf, n)) and corner_dev(win.chain(win.x0), G, w, h) > 1.0
    x, c0, c1, acc = solve(win, 50)
    err = corner_dev(win.chain(x), G, w, h)
    assert err < 1e-9, (kind, cost, err, c0, c1, acc)
    assert c1 <= c0 and acc >= 1


@pytest.mark.parametrize("cost", [MOSAIC, TRANSFER])
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_fixed_restatement_reaches_the_least_squares_minimum(kind, cost):
    """Noisy correspondences and fixed poses a few pixels off the truth: the minimum over the free frames."""
    from scipy.optimize import least_squares
    w, h, n, span, nf = 640, 480, 8, 2, 2
    Wc, solve = WINDOWS[cost]
    G, arrs = window_arrays(kind, n, span, w, h, 80, 50 + kind, noise=0.5, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.array([(np.linalg.inv(G[t + d]) @ G[t]).reshape(-1) for t, d in links(n, span)])
    win = Wc(kind, n, span, w, h, *arrs, None, np.ones((L, 80), bool), H, np.tile([1, 80, 0], (L, 1)),
             F=shifted(G[:nf], 3.0, 5 + kind))
    x, _, _, _ = solve(win, 100)
    P = NPAR[kind]

    def fun(v):
        xx = win.x0.copy()
        xx[win.free] = v.reshape(-1, P)
        return win.residuals(xx).reshape(-1) / win.s

    ls = least_squares(fun, win.x0[win.free].reshape(-1), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=20000)
    xs = win.x0.copy()
    xs[win.free] = ls.x.reshape(-1, P)
    err = corner_dev(win.chain(x), win.chain(xs), w, h)
    assert err < 1e-6, (kind, cost, err)


@pytest.mark.parametrize("cost", [MOSAIC, TRANSFER])
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_one_fixed_frame_is_the_window_on_its_own(kind, cost):
    w, h, n, span = 640, 480, 8, 3
    Wc, solve = WINDOWS[cost]
    base = {MOSAIC: Window, TRANSFER: TransferWindow}[cost]
    G, arrs = window_arrays(kind, n, span, w, h, 60, 30 + kind, noise=0.5, outliers=0.0, dtype=np.float64)
    L = n_links(n, span)
    H = np.array([(np.linalg.inv(G[t + d]) @ G[t]).reshape(-1) for t, d in links(n, span)])
    args = (kind, n, span, w, h, *arrs, None, np.ones((L, 60), bool), H, np.tile([1, 60, 0], (L, 1)))
    a, b = base(*args), Wc(*args, F=np.eye(3)[None])
    assert np.array_equal(a.x0, b.x0) and a.used == b.used and a.free == b.free and a.conn == b.conn
    ra, rb = solve(a, 20), solve(b, 20)
    assert np.array_equal(ra[0], rb[0]) and ra[1:] == rb[1:]


# ---- on the device --------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _fixed(F, conn=None):
    return (_cu(np.asarray(F, np.float64).reshape(-1, 9)), None if conn is None else _cu(np.asarray(conn, np.int32)))


@pytest.mark.gpu
@pytest.mark.parametrize("nf", [2, 3])
@pytest.mark.parametrize("cost", [MOSAIC, TRANSFER])
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_fixed_adjustment_matches_the_restatement(nm, kind, cost, nf):
    """The 64-frame span-3 windows of test_adjustment_matches_the_restatement with frames 0 .. nf-1 fixed a few pixels
    off the truth: chain_out within 1e-3 px of the restatement, the chain place() rebuilds from H_out within 0.02 px,
    the report equal to the restatement's costs (never rising), and the fixed frames' chain_out within 1e-9 px of F."""
    w, h, n, span, thr = 640, 480, 64, 3, 4.0
    Wc, solve = WINDOWS[cost]
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 70 + kind)
    F = shifted(G[:nf], 3.0, 11 * nf + kind)
    H, st, chain, rep = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, iterations=10, cost=cost, fixed=_fixed(F))
    H, st, chain, rep = H.cpu().numpy(), st.cpu().numpy(), chain.cpu().numpy().reshape(n, 3, 3), rep.cpu().numpy()
    win = Wc(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy(), F=F)
    x, c0, c1, acc = solve(win, 10)
    ref = win.chain(x)
    err = corner_dev(chain, ref, w, h)
    placed = placed_chain(nm, torch.from_numpy(H).cuda(), torch.from_numpy(st).cuda(), w, h)
    perr = corner_dev(placed, ref, w, h)
    ferr = corner_dev(chain[:nf], F, w, h)
    pts = sum(len(a) for (a, _), u in zip(win.pts, win.used) if u)
    print(f"kind {kind}, cost {cost}, n_fixed {nf}: device vs restatement {err:.2e} px, placed chain {perr:.2e} px, fixed "
          f"frames {ferr:.2e} px, mean squared residual {rep[0]:.4f} -> {rep[1]:.4f} (restatement "
          f"{c0 / win.s ** 2 / pts:.4f} -> {c1 / win.s ** 2 / pts:.4f}), steps accepted {st[-1, 2]} / {acc}")
    assert err < 1e-3 and perr < 0.02 and ferr < 1e-9, (err, perr, ferr)
    assert rep[1] <= rep[0] and rep[2] == pts and rep[3] == sum(win.used)
    assert not any(u and t + d < nf for (t, d), u in zip(win.order, win.used))
    assert np.allclose(rep[:2], [c0 / win.s ** 2 / pts, c1 / win.s ** 2 / pts], rtol=1e-6)
    assert (st[:, 0] == 1).all()


# sha256 of H_out, status_out, chain_out and report_out of nm_ransac_adjust_chain_cost_f32(NM_ADJUST_TRANSFER) on the
# windows of _digest_window, as the build before fixed frames computed them (NVIDIA B200)
TRANSFER_DIGESTS = {0: "670d0792e1df0c8e2ed68637d86145acff481d50154300df7e1bc6259e2b7544",
                    1: "624cd111d31a1c0131e27411e3952da633920ce7cacb0971545e75945add7299",
                    2: "1fa46a6c7b64c9858a6dfa100976d8bf78e276202d4866d165a54318b58cb299"}


def _outs(n):
    return (torch.empty(n - 1, 9, device="cuda"), torch.empty(n - 1, 3, dtype=torch.int32, device="cuda"),
            torch.empty(n, 9, dtype=torch.float64, device="cuda"), torch.empty(4, dtype=torch.float64, device="cuda"))


def _call(nm, name, kind, cost, d_, span, mask, HL, SL, w, h, n, fixed=None, thr=4.0, it=10, out=None):
    """One call of nm_ransac_adjust_chain_cost_f32 (fixed None) or nm_ransac_adjust_chain_fixed_f32 (fixed = (n_fixed,
    chain pointer, conn pointer)); returns (rc, outputs)."""
    p = lambda t: C.c_void_p(t.data_ptr())
    out = out or _outs(n)
    mid = () if fixed is None else fixed
    rc = getattr(nm.load(), name)(kind, cost, *[p(a) for a in d_], d_[0].shape[1], None, d_[0].shape[1], thr, n, span, w, h,
                                  p(mask), p(HL), p(SL), *mid, it, *[p(o) for o in out], _stream())
    return rc, out


def _digest(out):
    return hashlib.sha256(b"".join(t.cpu().numpy().tobytes() for t in out)).hexdigest()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_one_fixed_frame_is_the_cost_entry(nm, kind):
    """n_fixed = 1 of the new entry (the arrays not read: a NaN chain and a zero conn) is bitwise
    nm_ransac_adjust_chain_cost_f32 for both costs, and both are bitwise what the build before fixed frames returned."""
    w, h, n, span, d_, HL, SL, mask = _digest_window(nm, kind)
    junk = (torch.full((1, 9), float("nan"), dtype=torch.float64, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda"))
    for cost, pinned in ((MOSAIC, MOSAIC_DIGESTS), (TRANSFER, TRANSFER_DIGESTS)):
        rc, old = _call(nm, "nm_ransac_adjust_chain_cost_f32", kind, cost, d_, span, mask, HL, SL, w, h, n)
        assert rc == 0
        for fx in ((1, None, None), (1, C.c_void_p(junk[0].data_ptr()), C.c_void_p(junk[1].data_ptr()))):
            rc, new = _call(nm, "nm_ransac_adjust_chain_fixed_f32", kind, cost, d_, span, mask, HL, SL, w, h, n, fixed=fx)
            assert rc == 0
            for a, b in zip(old, new):
                assert torch.equal(a, b), cost
        default = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, 4.0, cost=cost)
        for a, b in zip(old, default):
            assert torch.equal(a, b), cost
        digest = _digest(old)
        print(f"kind {kind}, cost {cost}: digest {digest}")
        assert digest == pinned[kind], (cost, digest)


@pytest.mark.gpu
def test_fixed_poses_are_rebased_and_disconnected(nm):
    """C_j = A F_j for an invertible A gives F_j's result; a singular C_0 disconnects every fixed frame j >= 1, which is
    bitwise fixed_conn = [1, 0, ...]; fixed_conn[j] = 0 drops frame j's links (the restatement's links and chain)."""
    kind, w, h, n, span, thr, nf = 2, 640, 480, 24, 3, 4.0, 3
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 170, npts=800)
    F = shifted(G[:nf], 2.0, 3)
    run = lambda C_, conn=None: nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=TRANSFER, fixed=_fixed(C_, conn))
    base = run(F)
    A = np.array([[1.6, 0.3, -50.0], [-0.2, 1.4, 30.0], [2e-5, -1e-5, 1.1]])
    moved = run(np.array([A @ f for f in F]))
    ch0, ch1 = (o[2].cpu().numpy().reshape(n, 3, 3) for o in (base, moved))
    assert corner_dev(ch0, ch1, w, h) < 1e-9
    assert corner_dev(placed_chain(nm, base[0], base[1], w, h), placed_chain(nm, moved[0], moved[1], w, h), w, h) < 1e-3
    sing = F.copy()
    sing[0] = np.diag([1.0, 1.0, 0.0])
    for C_ in (sing, np.where(np.arange(nf)[:, None, None] == 0, np.nan, F)):
        off = run(C_)
        ref = run(F, [1] + [0] * (nf - 1))
        for a, b in zip(off, ref):
            assert torch.equal(a, b)
    st = off[1].cpu().numpy()
    assert st[: nf - 1].tolist() == [[0, 0, 0]] * (nf - 1) and (st[nf - 1:, 0] == 1).all()
    conn = [1, 1, 0]
    H, st, chain, rep = run(F, conn)
    win = FixedTransferWindow(kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy(), F=F,
                              fconn=conn)
    assert win.conn[:nf] == [True, True, False] and sum(win.used) < sum(FixedTransferWindow(
        kind, n, span, w, h, *arrs, None, mask.cpu().numpy(), HL.cpu().numpy(), SL.cpu().numpy(), F=F).used)
    x, _, _, _ = transfer_restatement(win, 10)
    assert rep[3].item() == sum(win.used)
    assert st[1].tolist() == [0, 0, 0] and (st[2:, 0] == 1).all()
    assert corner_dev(chain.cpu().numpy().reshape(n, 3, 3), win.chain(x), w, h) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 2])
def test_fixed_adjustment_arguments_reproducibility_and_graph_capture(nm, kind):
    w, h, n, span, thr, nf = 640, 480, 24, 3, 4.0, 3
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, n, span, w, h, 140 + kind, npts=800)
    fx = _fixed(shifted(G[:nf], 2.0, 4), [1, 1, 1])
    out = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=TRANSFER, fixed=fx)
    again = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, cost=TRANSFER, fixed=fx)
    for a, b in zip(out, again):
        assert torch.equal(a, b)
    assert out[1][-1, 2].item() >= 1
    Hg, Sg = torch.empty_like(out[0]), torch.empty_like(out[1])
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg), cost=TRANSFER, fixed=fx)
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    Hg.zero_()
    Sg.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        _, _, cg, rg = nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, out=(Hg, Sg), cost=TRANSFER, fixed=fx)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(Hg, out[0]) and torch.equal(Sg, out[1]) and torch.equal(cg, out[2]) and torch.equal(rg, out[3])
    # argument checks
    pc, pk = C.c_void_p(fx[0].data_ptr()), C.c_void_p(fx[1].data_ptr())
    call = lambda f: _call(nm, "nm_ransac_adjust_chain_fixed_f32", kind, TRANSFER, d_, span, mask, HL, SL, w, h, n, fixed=f)[0]
    assert call((nf, pc, pk)) == 0 and call((nf, pc, None)) == 0 and call((1, None, None)) == 0
    for bad in ((0, pc, pk), (-1, pc, pk), (n, pc, pk), (n + 1, pc, pk), (2, None, pk), (nf, None, None)):
        assert call(bad) == -1, bad
    with pytest.raises(nm.NmError):
        nm.adjust_chain(kind, *d_, None, span, mask, HL, SL, w, h, thr, fixed=_fixed(np.tile(np.eye(3), (n, 1, 1))))
    torch.cuda.synchronize()


# ---- the stream pipeline ---------------------------------------------------------------------------------------------
def _eleven_frames(nm):
    from niftymatch_b200 import synth
    w, h = 512, 384
    base = synth.scene(w + 80, h + 80, synth.SEED_BASE + 9)
    offs = [(8 + 6 * k, 8 + 5 * k - (k % 3)) for k in range(11)]
    fr = _cu(np.stack([base[oy: oy + h, ox: ox + w] for ox, oy in offs]))
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    return w, h, len(offs), fr, nm.SiftBatch(P, 5, 8192)


KW = dict(kind=2, inlier_threshold=1.0, iterations=512, seed=5, refine_rounds=1, span=3)


@pytest.mark.gpu
@pytest.mark.parametrize("O", [2, 3])
def test_stream_registrar_overlap_equals_the_public_calls(nm, O):
    """StreamRegistrar(span=3, overlap=O) over the 11-frame stream of test_stream_registrar_span_equals_the_public_calls
    (chunk 5) equals, bitwise, the public calls composed by hand: windows at 0, then at the previous end minus O, each
    anchored on the previous window's last O chain rows and connected flags, writing the pairs of its free frames.
    overlap=1 equals the default."""
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n, fr, sb = _eleven_frames(nm)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    for bad in (dict(KW, span=2, overlap=3), dict(KW, chunk=4, overlap=3), dict(KW, overlap=0)):
        with pytest.raises(ValueError):
            StreamRegistrar(sb, **dict(dict(chunk=5), **bad))
    H0, s0 = StreamRegistrar(sb, chunk=5, **KW).run(frames_of, 0, n)
    H1, s1 = StreamRegistrar(sb, chunk=5, overlap=1, **KW).run(frames_of, 0, n)
    assert torch.equal(H0, H1) and torch.equal(s0, s1)
    Ho, so = StreamRegistrar(sb, chunk=5, overlap=O, **KW).run(frames_of, 0, n)
    Hr, sr = torch.zeros_like(Ho), torch.zeros_like(so)
    c0, anchor, starts = 0, None, []
    while True:
        c1 = min(n, c0 + 5)
        m = c1 - c0
        S = min(3, m - 1)
        starts.append(c0)
        sb.run(frames_of(c0, c1))
        r = sb.results()
        cnt = r["counts"][:m]
        mt = nm.match_pairs_span(r["desc"][:m], cnt, S, 0.8)
        corr = nm.align_pairs_span(r["x"][:m], r["y"][:m], mt, cnt, S)
        HL, SL = [], []
        for d in range(1, S + 1):
            r0 = link_row(m, 0, d)
            a, b = nm.ransac_batch(2, *[c[r0: r0 + m - d] for c in corr], cnt[: m - d], 1.0, 512, 5 + c0 + ((d - 1) << 40))
            HL.append(a)
            SL.append(b)
        lc = torch.cat([cnt[: m - d] for d in range(1, S + 1)])
        HL, SL, mk = nm.refine_batch(2, *corr, lc, torch.cat(HL), torch.cat(SL), 1.0, 1)
        Ha, Sa, ch, _ = nm.adjust_chain(2, *corr, lc, S, mk, HL, SL, w, h, 1.0, 10, fixed=anchor)
        a = 0 if anchor is None else O - 1
        Hr[c0 + a: c1 - 1], sr[c0 + a: c1 - 1] = Ha[a:], Sa[a:]
        anchor = (ch[m - O:].contiguous(), Sa[m - O - 1: m - 1, 0].contiguous())
        if c1 == n:
            break
        c0 = c1 - O
    sb.close()
    assert starts == {2: [0, 3, 6], 3: [0, 2, 4, 6]}[O]
    assert torch.equal(Ho, Hr) and torch.equal(so, sr)
    assert (so[:, 0] == 1).all()


@pytest.mark.gpu
@pytest.mark.parametrize("O", [2, 3])
def test_resumed_run_equals_one_call(nm, O):
    """run(0, b) then run(b - O, n, resume=True) is bitwise run(0, n) when b ends a window of the single call; the first
    O - 1 rows of the resumed call are the previous call's.  A resume at another lo is refused."""
    from niftymatch_b200.dist import StreamRegistrar
    w, h, n, fr, sb = _eleven_frames(nm)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    reg = StreamRegistrar(sb, chunk=5, overlap=O, **KW)
    Hf, sf = reg.run(frames_of, 0, n)
    b = {2: 8, 3: 7}[O]
    Ha, sa = reg.run(frames_of, 0, b)
    with pytest.raises(ValueError):
        reg.run(frames_of, b - O + 1, n, resume=True)
    Hb, sb_ = reg.run(frames_of, b - O, n, resume=True)
    with pytest.raises(ValueError):
        StreamRegistrar(sb, chunk=5, overlap=O, **KW).run(frames_of, 0, n, resume=True)
    sb.close()
    assert torch.equal(Ha, Hf[: b - 1]) and torch.equal(sa, sf[: b - 1])
    assert torch.equal(Hb, Hf[b - O:]) and torch.equal(sb_, sf[b - O:])


# ---- windows of one synthetic stream ---------------------------------------------------------------------------------
def stream_windows(nm, kind, d_, HL, SL, mask, N, span, chunk, O, w, h, cost=TRANSFER, thr=4.0):
    """adjust_chain over the windows StreamRegistrar(chunk, span, overlap=O) forms on a stream whose links (span layout
    of all N frames) are given: each window's rows sliced out of the stream's.  Returns (frame -> frame-0 chain (N, 3, 3)
    float64, sum of report[3], all frames connected)."""
    rows_of = lambda c0, m, S: torch.tensor([link_row(N, c0 + t, d) for t, d in links(m, S)], device="cuda")
    Gg = [np.eye(3)]
    c0, anchor, used, conn = 0, None, 0.0, True
    chains, reps, stats = [], [], []
    while True:
        c1 = min(N, c0 + chunk)
        m = c1 - c0
        S = min(span, m - 1)
        rows = rows_of(c0, m, S)
        sel = lambda t: t.index_select(0, rows).contiguous()
        _, st, ch, rep = nm.adjust_chain(kind, *[sel(a) for a in d_], None, S, sel(mask), sel(HL), sel(SL), w, h, thr, cost=cost,
                                         fixed=anchor if O > 1 else None)
        chains.append((c0, ch))
        reps.append(rep)
        stats.append(st)
        anchor = (ch[m - O:], st[m - O - 1: m - 1, 0].contiguous())
        if c1 == N:
            break
        c0 = c1 - O
    for (c0, ch), rep, st in zip(chains, reps, stats):
        ch = ch.cpu().numpy().reshape(-1, 3, 3)
        for j in range(len(Gg) - c0, len(ch)):
            Gg.append(Gg[c0] @ ch[j])
        used += rep[3].item()
        conn = conn and bool((st[:, 0] == 1).all())
    return np.array(Gg), used, conn


@pytest.mark.gpu
def test_every_link_is_used_once(nm):
    """Windows of one synthetic 40-frame span-3 stream (chunk 8): with overlap = span the links used over all windows are
    the stream's usable links, each once; with overlap 1 the links that cross a window boundary are lost."""
    kind, w, h, N, span, chunk = 2, 640, 480, 40, 3, 8
    G, arrs, d_, HL, SL, mask = device_window(nm, kind, N, span, w, h, 200, npts=400)
    usable = ((SL[:, 0] == 1) & (mask.sum(1) >= MINPTS[kind])).cpu().numpy()
    _, used3, conn3 = stream_windows(nm, kind, d_, HL, SL, mask, N, span, chunk, 3, w, h)
    _, used1, conn1 = stream_windows(nm, kind, d_, HL, SL, mask, N, span, chunk, 1, w, h)
    ends = list(range(chunk - 1, N - 1, chunk - 1))           # the frames overlap-1 windows share
    inside = sum(1 for (t, d), u in zip(links(N, span), usable) if u and not any(t < e < t + d for e in ends))
    print(f"links used: overlap 3 {used3:.0f}, overlap 1 {used1:.0f}, usable {int(usable.sum())}, inside windows of overlap 1 {inside}")
    assert conn3 and conn1
    assert used3 == usable.sum() > 0.9 * n_links(N, span)
    assert used1 == inside < used3


def _last_corner_sq(Gk, Gt, w, h):
    c = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float64)
    return float((((map_pts(Gk, c) - map_pts(Gt, c)) ** 2).sum(1)).mean())


def drift_ratio(nm, kind, streams, N=120, chunk=8, span=3, w=640, h=480, npts=200, O=3):
    """Mean over `streams` synthetic streams of the last frame's mean squared corner error, overlap 1 and O."""
    e = {1: [], O: []}
    for s in range(streams):
        G, arrs, d_, HL, SL, mask = device_window(nm, kind, N, span, w, h, 1000 + 7 * s + kind, npts=npts, rounds=2)
        for o in (1, O):
            Gg, _, conn = stream_windows(nm, kind, d_, HL, SL, mask, N, span, chunk, o, w, h)
            assert conn
            e[o].append(_last_corner_sq(Gg[-1], G[-1], w, h))
    return float(np.mean(e[1])), float(np.mean(e[O]))


@pytest.mark.gpu
def test_overlap_lowers_the_drift_of_small_windows(nm):
    """64 synthetic translation streams of 120 frames (200 correspondences per link, sigma 0.3 px, 30 % outliers), 8-frame
    windows, span 3, transfer cost: the mean squared last-frame corner error with overlap 3 is below overlap 1 (a 1-D
    model of equal-noise links predicts a ratio of 0.64, and 0.90 is the 99.9th percentile of that ratio over 64 streams).
    The similarity and homography ratios (16 streams each) and the worst corner error of the 24-frame SIFT crop stream
    (homography, chunk 8) at overlap 1 and 3 are printed."""
    from niftymatch_b200.dist import StreamRegistrar
    e1, e3 = drift_ratio(nm, 0, 64)
    print(f"translation, 64 streams: last frame mean squared corner error, overlap 1 {e1:.3e} px^2, overlap 3 {e3:.3e} px^2, "
          f"ratio {e3 / e1:.3f}")
    for kind in (1, 2):
        a, b = drift_ratio(nm, kind, 16)
        print(f"kind {kind}, 16 streams: overlap 1 {a:.3e} px^2, overlap 3 {b:.3e} px^2, ratio {b / a:.3f}")
    w, h, n, offs, bgra = _crop_stream()
    fr = torch.from_numpy(bgra).cuda()
    P = nm.SiftParams(w, h)
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 8, 8192)
    frames_of = lambda t0, t1: fr[t0:t1].contiguous()
    for cost in (MOSAIC, TRANSFER):
        errs = {}
        for O in (1, 3):
            reg = StreamRegistrar(sb, chunk=8, kind=nm.HOMOGRAPHY, inlier_threshold=0.25, iterations=512, seed=3, refine_rounds=2,
                                  span=3, adjust_cost=cost, overlap=O)
            H, st = reg.run(frames_of, 0, n)
            assert (st[:, 0] == 1).all()
            errs[O] = _stream_errors(nm, H, st, w, h, offs)
        print(f"homography crop stream, cost {cost}, worst corner error: overlap 1 {errs[1]:.3f} px, overlap 3 {errs[3]:.3f} px")
    sb.close()
    assert e3 < e1, (e1, e3)
