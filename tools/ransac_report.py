"""Registration parity report on a GPU box: product (C-ABI) vs the reference's kernels (oracle/_ref) vs the CPU
oracle on the fixture scene of tests/_util.py (development aid).

--refine: the refit leg instead (nm_ransac_refine_batch_f32): time of the batched RANSAC alone and followed by 1 or 2
refit rounds (64 pairs x 8 192 correspondences, 70 % inliers, 1 024 hypotheses; CUDA events, the three variants in
alternating windows), corner error against the ground truth of the RANSAC model, the refit and a float64 fit to the
true inliers, and the 2 048-frame 1080p StreamRegistrar rate of bench.py with refine_rounds 0 and 2.

--adjust: the skip-link leg (nm_match_pairs_span_f32 ... nm_ransac_adjust_chain_cost_f32): time per 64-frame 1080p
window of each stage at span 1, 2, 3 (the frames of bench.py's stream, CUDA events, the spans in alternating windows),
the adjustment with the mosaic and the transfer cost, the 2 048-frame 1080p StreamRegistrar rate at span 1, 2, 3 with
refine_rounds 0 and 2 (span 3 with either cost), and the last frame's corner error on the synthetic 64-frame windows of
tests/test_gpu_chain_adjust.py for chained span-1 refits and the span-2 / span-3 adjustment with either cost.

--adjust --overlap O: the window-overlap leg instead (StreamRegistrar(span=3, overlap=O), adjust_chain(fixed=...)):
time per 64-frame and per 8-frame 1080p window (the five public calls, transfer cost) unanchored against anchored on O
fixed frames, in alternating windows; the 2 048-frame 1080p StreamRegistrar rate at span 3 (transfer cost, two refit
rounds) with overlap 1 and O; and the drift figures of tests/test_gpu_chain_adjust_fixed.py (synthetic 120-frame
streams in 8-frame windows, the SIFT crop stream) with overlap 1 and O."""
import os
import subprocess
import sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import niftymatch_b200 as nm  # noqa: E402


def refine_leg():
    import bench
    from tests.test_gpu_ransac_refine import scene, true_model, fit_homography, corner_error
    from niftymatch_b200.dist import StreamRegistrar
    stream_np = bench.render_frames(bench.stream_jobs(0, 32))
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card)
    rng = np.random.default_rng(12)
    n_pairs, n, thr = 64, 8192, 4.0
    arrs = [np.empty((n_pairs, n), np.float32) for _ in range(4)]
    truth, floor = [], []
    for p in range(n_pairs):
        Ht = true_model(2, rng)
        sc = scene(Ht, n, rng)
        for a, v in zip(arrs, sc[:4]):
            a[p] = v
        m = sc[4]
        floor.append(corner_error(fit_homography(np.stack([sc[0][m], sc[1][m]], 1).astype(np.float64),
                                                 np.stack([sc[2][m], sc[3][m]], 1).astype(np.float64)), Ht))
        truth.append(Ht)
    d = [torch.from_numpy(a).cuda() for a in arrs]
    H, st = nm.ransac_batch(2, *d, None, thr, 1024, 1)
    outs = {r: nm.refine_batch(2, *d, None, H, st, thr, rounds=r) for r in (1, 2)}
    Hn, stn = H.cpu().numpy(), st.cpu().numpy()
    rows = [("RANSAC model", [corner_error(Hn[p], truth[p]) for p in range(n_pairs)])]
    for r in (1, 2):
        Hr = outs[r][0].cpu().numpy()
        rows.append((f"refined, rounds = {r}", [corner_error(Hr[p], truth[p]) for p in range(n_pairs)]))
        print(f"rounds {r}: refits kept {np.bincount(outs[r][1][:, 2].cpu().numpy()).tolist()}, inliers "
              f"{stn[:, 1].sum()} -> {int(outs[r][1][:, 1].sum())}")
    rows.append(("float64 fit to the true inliers", floor))
    for name, e in rows:
        e = np.array(e)
        print(f"corner error, {name}: mean {e[:, 1].mean():.4f} px, max {e[:, 0].max():.4f} px")

    def run(rounds):
        H, st = nm.ransac_batch(2, *d, None, thr, 1024, 1)
        if rounds:
            nm.refine_batch(2, *d, None, H, st, thr, rounds=rounds, out=(H, st))
    for r in (0, 1, 2):
        for _ in range(3):
            run(r)
    torch.cuda.synchronize()
    times = {0: [], 1: [], 2: []}
    for _ in range(8):
        for r in (0, 1, 2):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                run(r)
            e1.record()
            torch.cuda.synchronize()
            times[r].append(e0.elapsed_time(e1) / 10 * 1e3)
    for r in (0, 1, 2):
        t = np.array(times[r])
        print(f"nm_ransac_batch_f32{'' if r == 0 else f' + refine rounds = {r}'}: median {np.median(t):.0f} us "
              f"(windows {t.min():.0f} - {t.max():.0f}); refine share {np.median(t) - np.median(times[0]):.0f} us")
    # the stream leg of bench.py on one GPU, with and without the refit
    P = nm.SiftParams(bench.W, bench.H)
    sb = nm.SiftBatch(P, bench.BATCH, bench.CAPACITY)
    base = torch.from_numpy(stream_np).cuda()
    frames_of = lambda t0, t1: base.index_select(0, torch.arange(t0, t1, device="cuda") % base.shape[0])
    n_stream = 2048
    for rep in range(2):
        for rounds in (0, 2):
            reg = StreamRegistrar(sb, chunk=sb.max_batch, refine_rounds=rounds)
            reg.run(frames_of, 0, sb.max_batch + 1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            Hs, sts = reg.run(frames_of, 0, n_stream)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            print(f"stream {n_stream} frames 1080p, refine_rounds {rounds}: {n_stream / ms * 1e3:.0f} frames/s "
                  f"({ms:.1f} ms), registered pairs {int((sts[:, 0] == 1).sum())}")
    sb.close()


def _card():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True).stdout.strip()
    print("card:", card)


def adjust_leg():
    import bench
    from niftymatch_b200.dist import StreamRegistrar
    from niftymatch_b200.match import link_row
    from niftymatch_b200.synth import map_points, span_window
    _card()
    stream_np = bench.render_frames(bench.stream_jobs(0, 32))
    P = nm.SiftParams(bench.W, bench.H)
    sb = nm.SiftBatch(P, bench.BATCH, bench.CAPACITY)
    base = torch.from_numpy(stream_np).cuda()
    frames_of = lambda t0, t1: base.index_select(0, torch.arange(t0, t1, device="cuda") % base.shape[0])
    # stages of one 64-frame window
    n, kind, thr, iters = sb.max_batch, 2, 4.0, 1024
    sb.run(frames_of(0, n))
    r = sb.results()
    cnt = r["counts"][:n]
    state = {}

    def stage(span, name):
        if name == "match":
            state["m"] = nm.match_pairs_span(r["desc"][:n], cnt, span, 0.8)
        elif name == "align":
            state["c"] = nm.align_pairs_span(r["x"][:n], r["y"][:n], state["m"], cnt, span)
        elif name == "ransac":
            out = [nm.ransac_batch(kind, *[c[link_row(n, 0, d): link_row(n, 0, d) + n - d] for c in state["c"]], cnt[: n - d], thr,
                                   iters, (d - 1) << 40) for d in range(1, span + 1)]
            state["H"], state["S"] = torch.cat([o[0] for o in out]), torch.cat([o[1] for o in out])
            state["lc"] = torch.cat([cnt[: n - d] for d in range(1, span + 1)])
        elif name == "refine":
            state["H"], state["S"], state["k"] = nm.refine_batch(kind, *state["c"], state["lc"], state["H"], state["S"], thr, 2)
        else:
            nm.adjust_chain(kind, *state["c"], state["lc"], span, state["k"], state["H"], state["S"], bench.W, bench.H, thr,
                            cost=nm.TRANSFER if name == "adjust (transfer)" else nm.MOSAIC)
    names = ("match", "align", "ransac", "refine", "adjust", "adjust (transfer)")
    times = {(s, k): [] for s in (1, 2, 3) for k in names}
    for rep in range(6):
        for span in (1, 2, 3):
            for k in names:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                stage(span, k)
                e1.record()
                torch.cuda.synchronize()
                if rep >= 1:
                    times[(span, k)].append(e0.elapsed_time(e1))
    for span in (1, 2, 3):
        tot = sum(np.median(times[(span, k)]) for k in names[:-1])
        print(f"span {span}, one 64-frame 1080p window: " + ", ".join(f"{k} {np.median(times[(span, k)]):.2f} ms" for k in names)
              + f"; sum with the mosaic cost {tot:.2f} ms")
    # the stream leg of bench.py
    n_stream = 2048
    for rep in range(2):
        for span, cost in ((1, nm.MOSAIC), (2, nm.MOSAIC), (3, nm.MOSAIC), (3, nm.TRANSFER)):
            for rounds in (0, 2):
                reg = StreamRegistrar(sb, chunk=sb.max_batch, refine_rounds=rounds, span=span, adjust_cost=cost)
                reg.run(frames_of, 0, sb.max_batch + 1)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                Hs, sts = reg.run(frames_of, 0, n_stream)
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1)
                print(f"stream {n_stream} frames 1080p, span {span}{' (transfer cost)' if cost else ''}, refine_rounds {rounds}: "
                      f"{n_stream / ms * 1e3:.0f} frames/s "
                      f"({ms:.1f} ms), connected pairs {int((sts[:, 0] == 1).sum())}")
    sb.close()
    # synthetic accuracy: windows of synth.span_window through RANSAC per d (link seeds as StreamRegistrar) and 2 refits
    w, h, n, thr = 640, 480, 64, 4.0
    c = np.array([[0, 0], [w - 1, 0], [0, h - 1], [w - 1, h - 1]], np.float64)
    for kind in (0, 1, 2):
        e = {1: [], (2, 0): [], (3, 0): [], (2, 1): [], (3, 1): []}
        for wnd in range(4):
            seed = 90 + 10 * wnd + kind
            G, arrs = span_window(kind, n, 3, w, h, 2000, seed)
            d_ = [torch.from_numpy(a).cuda() for a in arrs]
            out = [nm.ransac_batch(kind, *[a[link_row(n, 0, d): link_row(n, 0, d) + n - d] for a in d_], None, thr, 512,
                                   seed + ((d - 1) << 40)) for d in (1, 2, 3)]
            HL, SL, mask = nm.refine_batch(kind, *d_, None, torch.cat([o[0] for o in out]), torch.cat([o[1] for o in out]), thr, 2)
            last = lambda Gk: np.hypot(*(map_points(Gk[-1], c) - map_points(G[-1], c)).T).mean()
            e[1].append(last(nm.place(HL[: n - 1].contiguous(), SL[: n - 1].contiguous(), w, h).chain.cpu().numpy().reshape(n, 3, 3)))
            for span in (2, 3):                  # the span-2 layout is the first rows of the span-3 one
                L = span * n - span * (span + 1) // 2
                for cost in (nm.MOSAIC, nm.TRANSFER):
                    _, _, chain, _ = nm.adjust_chain(kind, *[a[:L] for a in d_], None, span, mask[:L], HL[:L], SL[:L], w, h, thr,
                                                     cost=cost)
                    e[span, cost].append(last(chain.cpu().numpy().reshape(n, 3, 3)))
        m = {k: float(np.mean(v)) for k, v in e.items()}
        for cost, name in ((nm.MOSAIC, "mosaic"), (nm.TRANSFER, "transfer")):
            print(f"synthetic 64-frame windows (4), kind {kind}, {name} cost: last frame mean corner error, chained span-1 "
                  f"refits {m[1]:.4f} px, span 2 {m[2, cost]:.4f} px ({m[2, cost] / m[1]:.3f}), span 3 {m[3, cost]:.4f} px "
                  f"({m[3, cost] / m[1]:.3f})")


def overlap_leg(O):
    import bench
    from niftymatch_b200.dist import StreamRegistrar, adjust_window
    from tests.test_gpu_chain_adjust import _crop_stream, _stream_errors
    from tests.test_gpu_chain_adjust_fixed import drift_ratio
    _card()
    stream_np = bench.render_frames(bench.stream_jobs(0, 32))
    P = nm.SiftParams(bench.W, bench.H)
    sb = nm.SiftBatch(P, bench.BATCH, bench.CAPACITY)
    base = torch.from_numpy(stream_np).cuda()
    frames_of = lambda t0, t1: base.index_select(0, torch.arange(t0, t1, device="cuda") % base.shape[0])
    span, kind, thr, iters = 3, 2, 4.0, 1024
    sb.run(frames_of(0, sb.max_batch))
    r = sb.results()
    for n in (sb.max_batch, 8):
        win = lambda fixed: adjust_window(r, n, span, bench.W, bench.H, kind, 0.8, thr, iters, 0, 2, None, adjust_cost=nm.TRANSFER,
                                          fixed=fixed)
        fixed = (win(None)[2][:O].contiguous(), None)            # frames 0 .. O-1 at their adjusted poses
        times = {1: [], O: []}
        for rep in range(7):
            for o in (1, O):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                win(None if o == 1 else fixed)
                e1.record()
                torch.cuda.synchronize()
                if rep >= 1:
                    times[o].append(e0.elapsed_time(e1))
        print(f"one {n}-frame 1080p window (match, align, RANSAC, refit, adjust; transfer cost): " + ", ".join(
            f"overlap {o} {np.median(times[o]):.2f} ms (windows {min(times[o]):.2f} - {max(times[o]):.2f}), "
            f"{np.median(times[o]) / (n - o):.3f} ms per new frame" for o in (1, O)))
    n_stream = 2048
    for rep in range(2):
        for o in (1, O):
            reg = StreamRegistrar(sb, chunk=sb.max_batch, refine_rounds=2, span=span, adjust_cost=nm.TRANSFER, overlap=o)
            reg.run(frames_of, 0, sb.max_batch + 1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            Hs, sts = reg.run(frames_of, 0, n_stream)
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1)
            print(f"stream {n_stream} frames 1080p, span 3 (transfer cost), refine_rounds 2, overlap {o}: "
                  f"{n_stream / ms * 1e3:.0f} frames/s ({ms:.1f} ms), connected pairs {int((sts[:, 0] == 1).sum())}")
    sb.close()
    for kind, streams in ((0, 64), (1, 16), (2, 16)):
        a, b = drift_ratio(nm, kind, streams, O=O)
        print(f"synthetic 120-frame streams ({streams}), kind {kind}, 8-frame windows, span 3, transfer cost: last frame mean "
              f"squared corner error, overlap 1 {a:.3e} px^2, overlap {O} {b:.3e} px^2, ratio {b / a:.3f}")
    w, h, n, offs, bgra = _crop_stream()
    fr = torch.from_numpy(bgra).cuda()
    Pc = nm.SiftParams(w, h)
    Pc._peak_threshold = 2.0
    sbc = nm.SiftBatch(Pc, 8, 8192)
    for cost in (nm.MOSAIC, nm.TRANSFER):
        errs = {}
        for o in (1, O):
            reg = StreamRegistrar(sbc, chunk=8, kind=nm.HOMOGRAPHY, inlier_threshold=0.25, iterations=512, seed=3, refine_rounds=2,
                                  span=3, adjust_cost=cost, overlap=o)
            H, st = reg.run(lambda t0, t1: fr[t0:t1].contiguous(), 0, n)
            errs[o] = _stream_errors(nm, H, st, w, h, offs)
        print(f"24-frame SIFT crop stream, homography, chunk 8, span 3, {'transfer' if cost else 'mosaic'} cost: worst corner "
              f"error, overlap 1 {errs[1]:.3f} px, overlap {O} {errs[O]:.3f} px")
    sbc.close()


if "--adjust" in sys.argv and "--overlap" in sys.argv:
    overlap_leg(int(sys.argv[sys.argv.index("--overlap") + 1]))
    sys.exit(0)
if "--adjust" in sys.argv:
    adjust_leg()
    sys.exit(0)
if "--refine" in sys.argv:
    refine_leg()
    sys.exit(0)
from tests._util import (load_oracle, load_reflib, ransac_scene, ransac_rand_lists, checker_ransac_hypotheses,  # noqa: E402
                         normalise_h)

orc, ref = load_oracle(), load_reflib()
sx, sy, dx, dy, Ht = ransac_scene()
cu = lambda a: torch.from_numpy(a).cuda()
for kind, rl in ransac_rand_lists(sx).items():
    Hp, ip = nm.ransac_hypotheses(kind, cu(sx), cu(sy), cu(dx), cu(dy), cu(rl), 4.0)
    Hp, ip = Hp.cpu().numpy(), ip.cpu().numpy()
    Ho, io = checker_ransac_hypotheses(orc.lib, "orc", kind, sx, sy, dx, dy, rl, 4.0)
    line = f"kind {kind}: product best {ip.max()}@{ip.argmax()}  oracle best {io.max()}@{io.argmax()}  |inl p-o| max {np.abs(ip - io).max()}"
    line += f"  H bitwise p==o {np.array_equal(Hp, Ho)}  |Hn p-o| max {np.abs(normalise_h(Hp) - normalise_h(Ho)).max():.3g}"
    if ref is not None:
        Hr, ir = checker_ransac_hypotheses(ref.lib, "nmref", kind, sx, sy, dx, dy, rl, 4.0)
        line += f"\n        reference best {ir.max()}@{ir.argmax()}  |inl p-r| max {np.abs(ip - ir).max()} (n diff {int((ip != ir).sum())})"
        line += f"  H bitwise p==r {np.array_equal(Hp, Hr)}  |Hn p-r| max {np.abs(normalise_h(Hp) - normalise_h(Hr)).max():.3g}"
        line += f"  |Hn o-r| max {np.abs(normalise_h(Ho) - normalise_h(Hr)).max():.3g} |inl o-r| max {np.abs(io - ir).max()}"
    print(line)
    for seed in (1, 2):
        H, st = nm.ransac(kind, cu(sx), cu(sy), cu(dx), cu(dy), 4.0, 2000, seed)
        H2, st2 = nm.ransac(kind, cu(sx), cu(sy), cu(dx), cu(dy), 4.0, 2000, seed)
        print("   full", seed, st.cpu().tolist(), "repeatable", torch.equal(H, H2) and torch.equal(st, st2),
              (H.cpu().numpy() / max(abs(float(H[8])), 1e-30)).round(5).tolist())
    if ref is not None:
        H9 = np.zeros(9, np.float32)
        import ctypes as C
        P = lambda v: v.ctypes.data_as(C.c_void_p)
        ok = ref.lib.nmref_ransac(kind, P(sx), P(sy), P(dx), P(dy), len(sx), C.c_float(4.0), 2000, P(H9))
        print("   reference full", ok, (H9 / max(abs(H9[8]), 1e-30)).round(5).tolist())
def timing():
    # timing
    n = 8192
    sx, sy, dx, dy, _ = ransac_scene(n=n, seed=9)
    a = [cu(v) for v in (sx, sy, dx, dy)]
    for kind in (0, 1, 2):
        for it in (1024, 4096):
            for _ in range(5):
                nm.ransac(kind, *a, 4.0, it, 1)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(10):
                nm.ransac(kind, *a, 4.0, it, 1)
            e1.record()
            torch.cuda.synchronize()
            print(f"nm_ransac_f32 kind {kind} n {n} iterations {it}: {e0.elapsed_time(e1) / 10 * 1e3:.1f} us")

    # batched: 64 frame pairs in one launch sequence
    npairs = 64
    arrs = [torch.stack([cu(ransac_scene(n=n, seed=100 + p)[k]) for p in range(npairs)]).contiguous() for k in range(4)]
    for kind in (0, 2):
        for _ in range(3):
            nm.ransac_batch(kind, *arrs, None, 4.0, 1024, 1)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            nm.ransac_batch(kind, *arrs, None, 4.0, 1024, 1)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        print(f"nm_ransac_batch_f32 kind {kind}: {npairs} pairs x {n} correspondences x 1024 hypotheses: {ms * 1e3:.0f} us = {ms * 1e3 / npairs:.1f} us per pair")


for rep in range(2):
    print("timing pass", rep)
    timing()
