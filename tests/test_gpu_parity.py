"""GPU suite: the CUDA product, called through the C-ABI (include/nm_b200.h), against the CPU
oracle on identical seeded inputs, against the golden vectors captured from the reference's
own CUDA code, and -- when oracle/_ref/libnmref.so is present -- against the reference itself.

Tolerances (BASELINE.json north_star): keypoint position <= 0.01 px, scale / orientation
<= 1e-3, recall >= 99 %, descriptor L2 <= 1e-3 relative, identical match indices.  Everything
that is integer / index / pure fp32-arithmetic work is held to BITWISE equality instead."""
import ctypes as C
import os

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from niftymatch_b200 import synth  # noqa: E402
from tests._util import GOLDEN, ang_diff, equal_at_stored  # noqa: E402

ORIENT_TOL = 1e-5          # rad; north_star allows 1e-3
DESC_REL_TOL = 2e-5        # relative L2; north_star allows 1e-3


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _gold(name):
    return np.load(os.path.join(GOLDEN, name))


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def run_product(nm, frames, peak=0.0, capacity=8192, exact=False, num_octaves=-1, dense_grad=True):
    """dense_grad: the whole gradient maps are read back below, so they are computed everywhere; the default of
    the product (only the blocks keypoint windows read) is covered by test_sparse_gradient_maps_*."""
    n, h, w = frames.shape
    P = nm.SiftParams(w, h)
    P._peak_threshold = peak
    if num_octaves > 0:
        P._num_octaves = num_octaves
    sb = nm.SiftBatch(P, n, capacity)
    sb.set_exact_descriptor(exact)
    sb.set_dense_gradients(dense_grad)
    sb.run(_cu(frames))
    torch.cuda.synchronize()
    out = [read_frame(sb, f, grad=True) for f in range(n)]
    sb.close()
    return out


def read_frame(sb, f, grad=False):
    """Frame f of the last run of `sb` as host arrays: results, all Gaussian levels and (grad=True) gradient maps."""
    r = sb.results()
    c = int(r["counts"][f].item())
    seg = r["seg_counts"][f].cpu().numpy()
    nk = min(int(seg.sum()), sb.capacity)
    out = {
        "n": c, "seg_counts": seg, "desc": r["desc"][f, :c].cpu().numpy(), "x": r["x"][f, :c].cpu().numpy(),
        "y": r["y"][f, :c].cpu().numpy(), "kpts": r["kpts"][f, :nk].cpu().numpy(),
        "orient": r["orient"][f, :nk].cpu().numpy(),
        "levels": [[sb.level(f, o, l).cpu().numpy() for l in range(6)] for o in range(sb.n_oct)],
    }
    if grad:
        out["grad"] = [np.stack([sb.grad(f, o, l).cpu().numpy() for l in range(3)]) for o in range(sb.n_oct)]
    return out


def assert_frame_matches(p, c, check_levels=True):
    """p: product, c: checker (oracle / reference) frame dictionaries."""
    assert np.array_equal(p["seg_counts"], c["seg_counts"])
    assert p["n"] == c["n"]
    if check_levels:
        for o in range(len(c["levels"])):
            for l in range(6):
                assert np.array_equal(p["levels"][o][l], c["levels"][o][l]), f"octave {o} level {l} not bitwise equal"
    assert np.array_equal(p["kpts"], c["kpts"]), "keypoints not bitwise equal"
    assert np.array_equal(p["orient"] < 0, c["orient"] < 0)
    ok = c["orient"] >= 0
    if ok.any():
        assert ang_diff(p["orient"][ok], c["orient"][ok]).max() <= ORIENT_TOL
    if c["n"]:
        rel = np.linalg.norm(p["desc"] - c["desc"], axis=1) / np.maximum(np.linalg.norm(c["desc"], axis=1), 1e-20)
        assert rel.max() <= DESC_REL_TOL, rel.max()
        assert np.array_equal(p["x"], c["x"]) and np.array_equal(p["y"], c["y"])


# ------------------------------------------------------------------ parameters, taps
def test_params_and_taps_vs_reference(nm):
    g = _gold("params_taps.npz")
    for key in g.files:
        if key.startswith("params_"):
            w, h = map(int, key[len("params_"):].split("x"))
            P = nm.SiftParams(w, h)
            got = np.array([P._num_octaves, P._sigma_k, P._sigma_0, P._sigma_d_0, P._base_smooth] + P._sigmas, np.float64)
            assert np.array_equal(got, g[key]), key
    P = nm.SiftParams(640, 480)
    for which in range(-1, 5):
        taps, r = nm.gaussian_taps(P._base_smooth if which < 0 else P._sigmas[which])
        assert np.array_equal(taps, g[f"taps_{which}"])


# ------------------------------------------------------------------ per-stage operators
def test_blur_vs_reference_golden(nm):
    from niftymatch_b200 import sift as S
    g = _gold("convolve_208x144.npz")
    taps = g["taps"]
    out = S.blur(_cu(g["image"]), _cu(taps), (len(taps) - 1) // 2)
    assert np.array_equal(out.cpu().numpy(), g["result"])


@pytest.mark.parametrize("shape", [(77, 131), (64, 128), (1, 5), (200, 33), (130, 260), (700, 300), (2304, 2560)])
@pytest.mark.parametrize("radius", list(range(1, 17)) + [17, 20, 45])
def test_blur_vs_oracle_bitwise(nm, oracle, shape, radius):
    """nm_blur_f32 at every radius the tiled kernels are instantiated for (1..16) and the generic two-pass blur above
    them, up to the reference's largest kernel (radius 45).  Odd widths take the tile kernel with plain loads, the
    other small shapes the TMA tile kernel, 2304 x 2560 (720 tiles, 740 strip chunks) the persistent tile-walking
    kernel; test_forced_strip_blur_parity_suite re-runs every case through the strip-walking kernel.  Bitwise against
    the oracle, and within the fp32 rounding bound of a float64 convolution: the taps are random and asymmetric, so
    that check pins the direction (out[x] = sum_k in[x + k] * taps[R - k]) and the zero border independently."""
    from scipy.ndimage import convolve1d
    from niftymatch_b200 import sift as S
    h, w = shape
    rng = np.random.default_rng(radius * 1000 + h)
    img = (rng.random((h, w)) * 255).astype(np.float32)
    taps = rng.random(2 * radius + 1).astype(np.float32)
    taps /= taps.sum()
    res, buf = np.zeros_like(img), np.zeros_like(img)
    oracle.lib.orc_convolve(res.ctypes.data_as(C.c_void_p), img.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p),
                            w, h, taps.ctypes.data_as(C.c_void_p), radius)
    scratch = torch.empty((h, w), dtype=torch.float32, device="cuda")
    out = S.blur(_cu(img), _cu(taps), radius, buffer=scratch).cpu().numpy()
    assert np.array_equal(out, res)
    t64 = taps.astype(np.float64)
    ref = convolve1d(convolve1d(img.astype(np.float64), t64, axis=1, mode="constant"), t64, axis=0, mode="constant")
    # two chains of 2R+1 fp32 multiply-adds over non-negative terms summing to <= max|img|
    assert np.abs(out - ref).max() <= 4 * (2 * radius + 1) * 2.0 ** -24 * np.abs(img).max()


def test_downsample_subtract_gradient_vs_oracle(nm, oracle):
    from niftymatch_b200 import sift as S
    img = synth.scene(150, 101, synth.SEED_BASE + 5)
    img2 = synth.scene(150, 101, synth.SEED_BASE + 6)
    d = S.downsample2(_cu(img)).cpu().numpy()
    assert np.array_equal(d, img[::2, ::2][:50, :75])
    s = S.subtract(_cu(img), _cu(img2)).cpu().numpy()
    assert np.array_equal(s, img - img2)
    g = S.gradient(_cu(img)).cpu().numpy()
    ref = np.zeros((101, 150, 2), np.float32)
    oracle.lib.orc_gradient(img.ctypes.data_as(C.c_void_p), ref.ctypes.data_as(C.c_void_p), 150, 101)
    assert np.array_equal(g[..., 0], ref[..., 0])
    assert ang_diff(g[..., 1], ref[..., 1]).max() <= 2e-6
    assert (g[0] == 0).all() and (g[-1] == 0).all() and (g[:, 0] == 0).all() and (g[:, -1] == 0).all()


def test_compat_operator_chain_vs_oracle(nm, oracle):
    """The per-octave operators the reference API is made of (dense keypoint map, collate,
    orientations, descriptors), driven like siftfunctions.cu does."""
    from niftymatch_b200 import sift as S
    img = synth.scene(256, 192, synth.SEED_BASE)
    c = oracle.sift_frame(img, peak=0.0, want_grad=True)
    P = nm.SiftParams(256, 192)
    lv = [_cu(c["levels"][0][l]) for l in range(6)]
    dog = [S.subtract(lv[i + 1], lv[i]) for i in range(5)]
    grads = torch.stack([S.gradient(lv[i + 1]) for i in range(3)]).contiguous()
    off, items = 0, 0
    for l in range(3):
        dense = S.keypoints_dense(dog[l + 1], dog[l], dog[l + 2], 0.0, P._edge_threshold, 1.0, P._sigma_0, 3, l)
        kp = S.collate(dense)
        n = int(c["seg_counts"][l])
        assert kp.shape[0] == n
        assert np.array_equal(kp.cpu().numpy(), c["kpts"][off: off + n])
        ori = S.orientations(kp.contiguous(), grads, 256, 192, 1.0)
        co = c["orient"][off: off + n]
        assert np.array_equal(ori.cpu().numpy() < 0, co < 0)
        assert ang_diff(ori.cpu().numpy()[co >= 0], co[co >= 0]).max() <= ORIENT_TOL
        desc, x, y = S.descriptors(kp.contiguous(), ori, grads, 256, 192, 3, 1.0)
        cd = c["desc"][items: items + n]
        rel = np.linalg.norm(desc.cpu().numpy() - cd, axis=1) / np.maximum(np.linalg.norm(cd, axis=1), 1e-20)
        assert rel.max() <= DESC_REL_TOL
        assert np.array_equal(x.cpu().numpy(), c["x"][items: items + n])
        off += n
        items += n


# ------------------------------------------------------------------ batched SIFT
@pytest.mark.parametrize("name", ["sift_256x192.npz", "sift_384x256.npz"])
def test_sift_vs_reference_golden(nm, name):
    g = _gold(name)
    img = g["image"]
    for peak in (0.0, 2.0):
        tag = f"p{int(peak)}"
        p = run_product(nm, img[None], peak=peak)[0]
        assert np.array_equal(p["seg_counts"], g[f"{tag}_seg_counts"])
        assert np.array_equal(p["kpts"], g[f"{tag}_kpts"]), "keypoints not bitwise equal to the reference's"
        if peak == 0.0:
            n_oct = len(p["levels"])
            for o in range(n_oct):
                assert equal_at_stored(p["levels"][o][5], g[f"level5_oct{o}"])
                assert equal_at_stored(p["levels"][o][3], g[f"level3_oct{o}"])
            for l in range(6):
                assert np.array_equal(p["levels"][n_oct - 1][l], g[f"level{l}_oct{n_oct - 1}"])
            assert np.array_equal(p["grad"][n_oct - 1], g[f"grad_oct{n_oct - 1}"]), "gradient maps not bitwise equal"
        oi = g[f"{tag}_orient_in"]
        assert np.array_equal(p["orient"] < 0, oi < 0)
        assert ang_diff(p["orient"][oi >= 0], oi[oi >= 0]).max() <= ORIENT_TOL
        rd = g[f"{tag}_desc"]
        rel = np.linalg.norm(p["desc"] - rd, axis=1) / np.maximum(np.linalg.norm(rd, axis=1), 1e-20)
        assert rel.max() <= DESC_REL_TOL
        assert np.array_equal(p["x"], g[f"{tag}_x"]) and np.array_equal(p["y"], g[f"{tag}_y"])


def test_sift_vs_reference_public_orientation_kernel(nm):
    """The whole chain against reference-derived numbers with NO oracle in between: keypoints, the orientations of the
    reference's public kernel_orientations_optim (barriers hoisted so that it terminates on sm_70+, arithmetic
    untouched; tests/golden/README.md) and the descriptors the reference computed from ITS orientations."""
    g = _gold("sift_orient_public.npz")
    for (w, h, seed) in [(256, 192, synth.SEED_BASE), (384, 256, synth.SEED_BASE + 3)]:
        img = synth.scene(w, h, seed)
        for peak in (0.0, 2.0):
            tag = f"{w}x{h}_p{int(peak)}"
            p = run_product(nm, img[None], peak=peak)[0]
            assert np.array_equal(p["seg_counts"], g[f"{tag}_seg_counts"])
            assert np.array_equal(p["kpts"], g[f"{tag}_kpts"]), "keypoints not bitwise equal to the reference's"
            go = g[f"{tag}_orient"]
            assert np.array_equal(p["orient"] < 0, go < 0)
            assert ang_diff(p["orient"][go >= 0], go[go >= 0]).max() <= ORIENT_TOL
            gd = g[f"{tag}_desc"]
            assert p["n"] == len(gd)
            rel = np.linalg.norm(p["desc"] - gd, axis=1) / np.maximum(np.linalg.norm(gd, axis=1), 1e-20)
            assert rel.max() <= 1e-3, rel.max()
            assert np.array_equal(p["x"], g[f"{tag}_x"]) and np.array_equal(p["y"], g[f"{tag}_y"])


@pytest.mark.parametrize("size,peak", [((640, 480), 0.0), ((640, 480), 2.0), ((250, 130), 0.0), ((97, 161), 0.0)])
def test_sift_vs_oracle(nm, oracle, size, peak):
    w, h = size
    img = synth.scene(w, h, synth.SEED_BASE + w)
    p = run_product(nm, img[None], peak=peak)[0]
    c = oracle.sift_frame(img, peak=peak)
    assert_frame_matches(p, c)


def test_exact_and_fp32_descriptor_modes_agree(nm, oracle):
    img = synth.scene(384, 256, synth.SEED_BASE + 1)
    a = run_product(nm, img[None], exact=False)[0]
    b = run_product(nm, img[None], exact=True)[0]
    assert a["n"] == b["n"] > 100
    rel = np.linalg.norm(a["desc"] - b["desc"], axis=1) / np.linalg.norm(b["desc"], axis=1)
    assert rel.max() <= 5e-6
    c = oracle.sift_frame(img, want_levels=False)
    rel = np.linalg.norm(b["desc"] - c["desc"], axis=1) / np.linalg.norm(c["desc"], axis=1)
    assert rel.max() <= DESC_REL_TOL


def test_batch_frames_are_independent_and_ordered(nm, oracle):
    frames = np.stack([synth.scene(320, 200, synth.SEED_BASE + i) for i in range(3)] +
                      [np.zeros((200, 320), np.float32)])
    out = run_product(nm, frames, peak=0.0)
    for f in range(3):
        assert_frame_matches(out[f], oracle.sift_frame(frames[f]))
    assert out[3]["n"] == 0 and out[3]["seg_counts"].sum() == 0           # empty frame
    single = run_product(nm, frames[1:2])[0]
    assert np.array_equal(single["desc"], out[1]["desc"])                   # bit-reproducible, batch independent


def test_capacity_truncation_is_a_prefix(nm, oracle):
    img = synth.scene(256, 192, synth.SEED_BASE)
    full = run_product(nm, img[None], capacity=4096)[0]
    cut = run_product(nm, img[None], capacity=50)[0]
    assert cut["n"] == 50 and full["n"] > 50
    assert np.array_equal(cut["desc"], full["desc"][:50]) and np.array_equal(cut["x"], full["x"][:50])
    assert np.array_equal(cut["seg_counts"], full["seg_counts"])           # counts are pre-truncation
    c = oracle.sift_frame(img, capacity=50, want_levels=False)
    assert c["n"] == 50
    rel = np.linalg.norm(cut["desc"] - c["desc"], axis=1) / np.linalg.norm(c["desc"], axis=1)
    assert rel.max() <= DESC_REL_TOL


def test_early_return_rule(nm, oracle):
    img = np.full((96, 128), 128.0, np.float32)
    img[40:44, 60:64] += 50.0
    p = run_product(nm, img[None])[0]
    c = oracle.sift_frame(img)
    assert_frame_matches(p, c)


def test_forced_octave_count(nm, oracle):
    img = synth.scene(512, 384, synth.SEED_BASE + 2)
    p = run_product(nm, img[None], num_octaves=3)[0]
    c = oracle.sift_frame(img, num_octaves=3)
    assert_frame_matches(p, c)


def test_sift_vs_reference_library_direct(nm, reflib):
    """Same comparison against the reference's CUDA code running on this GPU (when built)."""
    img = synth.scene(640, 480, synth.SEED_BASE + 11)
    p = run_product(nm, img[None], peak=0.0)[0]
    r = reflib.sift_frame(img, peak=0.0, want_grad=True, orient_mode=2, orient_in=p["orient"])
    assert np.array_equal(p["seg_counts"], r["seg_counts"])
    for o in range(len(r["levels"])):
        for l in range(6):
            assert np.array_equal(p["levels"][o][l], r["levels"][o][l])
        assert np.array_equal(p["grad"][o], r["grad"][o])
    assert np.array_equal(p["kpts"], r["kpts"])
    rel = np.linalg.norm(p["desc"] - r["desc"], axis=1) / np.linalg.norm(r["desc"], axis=1)
    assert rel.max() <= DESC_REL_TOL


# ------------------------------------------------------------------ full-size properties
def test_1080p_batch_properties(nm):
    """At BASELINE.json's size the oracle is too slow to be the checker for a batch; use
    size-independent properties: duplicated frames give bit-identical results (determinism,
    batch independence), keypoint lists are raster-sorted inside each (octave, level) segment,
    seg_counts obey the early-return rule, counts = min(sum, capacity)."""
    base = synth.frame_batch(1920, 1080, 2)
    frames = np.stack([base[0], base[1], base[0], base[1]])
    n, cap = 4, 16384
    P = nm.SiftParams(1920, 1080)
    sb = nm.SiftBatch(P, n, cap)
    sb.run(_cu(frames))
    torch.cuda.synchronize()
    r = {k: v.cpu().numpy() for k, v in sb.results().items()}
    assert (r["counts"] > 1000).all()
    for a, b in ((0, 2), (1, 3)):
        c = r["counts"][a]
        assert c == r["counts"][b]
        assert np.array_equal(r["desc"][a, :c], r["desc"][b, :c])
        assert np.array_equal(r["kpts"][a, :c], r["kpts"][b, :c])
        assert np.array_equal(r["orient"][a, :c], r["orient"][b, :c])
    for f in range(2):
        seg = r["seg_counts"][f].reshape(-1, 3)
        assert r["counts"][f] == min(seg.sum(), cap)
        for row in seg:
            z = np.where(row == 0)[0]
            if len(z):
                assert (row[z[0]:] == 0).all()
        off = 0
        for o in range(seg.shape[0]):
            ow = 1920 >> o
            for l in range(3):
                k = r["kpts"][f, off: off + seg[o, l]]
                off += seg[o, l]
                if len(k) > 1:
                    assert (k[:, 3] == l).all()
    # run again: bit-identical (idempotent workspace reuse)
    sb.run(_cu(frames))
    torch.cuda.synchronize()
    r2 = sb.results()
    assert np.array_equal(r2["desc"].cpu().numpy()[0, : r["counts"][0]], r["desc"][0, : r["counts"][0]])
    sb.close()


def test_1080p_single_frame_vs_oracle(nm, oracle):
    """One full-size frame against the CPU oracle (about 3 s of CPU)."""
    img = synth.scene(1920, 1080, synth.SEED_BASE)
    p = run_product(nm, img[None], capacity=16384)[0]
    c = oracle.sift_frame(img, capacity=16384)
    assert_frame_matches(p, c)
    assert p["n"] > 5000


def test_1080p_batch_strip_blur_vs_oracle(nm, oracle):
    """Twenty 1080p frames = 300 column strips in octave 0: every octave-0 blur takes the streaming blur kernel
    (nm_pyramid.cu, blur_stream_kernel) oversubscribed with 4 CTAs per strip, each walking a quarter of the strip's
    16-row groups (the parts that start inside the strip after lead-in groups whose outputs are not stored).  First,
    a middle and the last frame against the CPU oracle, levels bitwise."""
    frames = np.stack([synth.scene(1920, 1080, synth.SEED_BASE + (i % 2)) for i in range(20)])
    out = run_product(nm, frames, capacity=16384)
    ref = [oracle.sift_frame(frames[f], capacity=16384) for f in (0, 1)]
    for f in (0, 9, 19):
        assert_frame_matches(out[f], ref[f % 2])


def test_stream_blur_piece_table_many_small_frames(nm, oracle):
    """800 frames of 128 x 199 = 800 one-strip launches for the streaming blur kernel (nm_pyramid.cu,
    blur_stream_kernel): with 740 persistent CTAs that is one round of whole strips plus 60 strips split into pieces
    shorter than a 16-row group (most CTAs get an empty piece, the others start inside a strip behind lead-in
    groups); the odd height exercises the last row of the decimated second output.  Sampled frames, all levels of
    both octaves bitwise against the CPU oracle."""
    w, h, n = 128, 199, 800
    scenes = [synth.scene(w, h, synth.SEED_BASE + 40 + i) for i in range(4)]
    frames = np.stack([scenes[i % 4] for i in range(n)])
    P = nm.SiftParams(w, h)
    sb = nm.SiftBatch(P, n, 2048)
    sb.run(_cu(frames))
    torch.cuda.synchronize()
    ref = [oracle.sift_frame(s, capacity=2048) for s in scenes]
    counts = sb.results()["counts"].cpu().numpy()
    assert np.array_equal(counts, np.array([ref[i % 4]["n"] for i in range(n)]))
    for f in (0, 1, 2, 3, 368, 369, 370, 738, 739, 740, 741, 742, 770, 797, 798, 799):
        for o in range(P._num_octaves):
            for l in range(6):
                assert np.array_equal(sb.level(f, o, l).cpu().numpy(), ref[f % 4]["levels"][o][l]), (f, o, l)
    sb.close()


def test_wide_blur_radius_in_the_batched_path(nm, oracle):
    """SiftParams members are mutable and the reference accepts kernels up to 91 taps (radius 45): a level sigma
    above 4 gives a radius above 16, which the tiled TMA blur does not cover -- the batched path then runs the generic
    two-pass blur through the context's row-pass buffer (nm_sift_create allocates it).  Every level must still be
    bitwise the oracle's convolution of the level below, and the run must produce keypoints."""
    w, h = 200, 150
    img = synth.scene(w, h, synth.SEED_BASE + 77)
    P = nm.SiftParams(w, h)
    P.c.sigmas[3] = 4.3            # radius 18
    P.c.sigmas[4] = 5.2            # radius 21
    sb = nm.SiftBatch(P, 2, 4096)
    sb.run(_cu(np.stack([img, img[::-1].copy()])))
    torch.cuda.synchronize()
    assert int(sb.results()["counts"][0].item()) > 20
    for f, im in enumerate((img, img[::-1].copy())):
        for lvl, sigma in ((4, 4.3), (5, 5.2)):
            taps, radius = nm.gaussian_taps(sigma)
            assert radius > 16
            src = sb.level(f, 0, lvl - 1).cpu().numpy().copy()
            res, buf = np.zeros_like(src), np.zeros_like(src)
            oracle.lib.orc_convolve(res.ctypes.data_as(C.c_void_p), src.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p),
                                    w, h, taps.ctypes.data_as(C.c_void_p), radius)
            assert np.array_equal(sb.level(f, 0, lvl).cpu().numpy(), res), (f, lvl)
    sb.close()


def test_sparse_gradient_maps_give_identical_results(nm):
    """Default mode: gradient maps only for the 8 x 32 blocks marked by emit_kernel from the keypoints' orientation
    and descriptor windows.  Keypoints, orientations, descriptors and coordinates must be BITWISE those of the
    dense-map run (same kernels reading the same samples), at both thresholds, on frames of several sizes, with
    stale data in the unmarked blocks (the context is reused: the maps hold the previous frame's values)."""
    for (w, h, peak) in [(256, 192, 0.0), (256, 192, 2.0), (640, 480, 0.0), (333, 250, 4.0)]:
        frames = np.stack([synth.scene(w, h, synth.SEED_BASE + 40 + i) for i in range(3)])
        P = nm.SiftParams(w, h)
        P._peak_threshold = peak
        sb = nm.SiftBatch(P, 3, 8192)
        res = {}
        for mode in ("dense", "sparse", "sparse_again"):
            sb.set_dense_gradients(mode == "dense")
            fr = frames if mode != "sparse_again" else frames[::-1].copy()      # other frames left their maps behind
            sb.run(_cu(fr))
            torch.cuda.synchronize()
            if mode == "sparse_again":
                sb.run(_cu(frames))
                torch.cuda.synchronize()
            r = sb.results()
            res[mode] = {k: r[k].cpu().numpy().copy() for k in ("counts", "kpts", "orient", "desc", "x", "y")}
        assert res["dense"]["counts"].min() > 0
        for mode in ("sparse", "sparse_again"):
            for f in range(3):
                c = int(res["dense"]["counts"][f])
                assert res[mode]["counts"][f] == c
                for k in ("kpts", "orient", "desc", "x", "y"):
                    assert np.array_equal(res[mode][k][f, :c], res["dense"][k][f, :c]), (w, h, peak, mode, f, k)
        sb.close()


@pytest.mark.parametrize("stream", ["1", "0"])
def test_forced_strip_blur_parity_suite(stream):
    """The strip-walking blur kernels are only chosen for large launches; NM_BLUR_STRIP_MIN=1 forces them for every
    TMA-describable source, and the blur / SIFT parity tests are re-run that way in a child process
    (ranges that start inside a strip, one-chunk strips, 1-row images, the decimated second output).
    stream=1: the SIFT pyramid takes blur_stream_kernel (warp-specialised) and nm_blur_f32 blur_strip_kernel;
    stream=0 (NM_BLUR_STREAM=0): blur_strip_kernel everywhere."""
    import subprocess
    import sys
    if os.environ.get("NM_BLUR_STRIP_MIN"):
        pytest.skip("already the forced run")
    env = dict(os.environ, NM_BLUR_STRIP_MIN="1", NM_BLUR_STREAM=stream)
    sel = ("test_blur_vs_oracle_bitwise or test_blur_vs_reference_golden or test_sift_vs_oracle or "
           "test_sift_vs_reference_golden or test_4k_six_octave or test_forced_octave_count")
    r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", "-p", "no:cacheprovider", __file__, "-k", sel],
                       env=env, capture_output=True, text=True, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


def test_run_host_end_to_end(nm, oracle):
    frames = np.stack([synth.scene(256, 192, synth.SEED_BASE + i) for i in range(2)])
    P = nm.SiftParams(256, 192)
    sb = nm.SiftBatch(P, 2, 1024)
    out = sb.run_host(frames)
    for f in range(2):
        c = oracle.sift_frame(frames[f], want_levels=False)
        n = int(out["counts"][f])
        assert n == c["n"]
        rel = np.linalg.norm(out["desc"][f, :n].numpy() - c["desc"], axis=1) / np.linalg.norm(c["desc"], axis=1)
        assert rel.max() <= DESC_REL_TOL
        assert np.array_equal(out["x"][f, :n].numpy(), c["x"])
    sb.close()


def test_masked_detector_batched_vs_reference_and_oracle(nm, oracle):
    """compute_keypoints_with_mask in the batched path (nm_sift_set_mask_image): keypoints bitwise the
    reference's (tests/golden, captured from compute_keypoints_with_mask on a B200) and the oracle's;
    descriptors within tolerance; removing the mask restores the unmasked result."""
    g = _gold("sift_256x192_masked.npz")
    img = g["image"]
    P = nm.SiftParams(256, 192)
    sb = nm.SiftBatch(P, 2, 4096)
    frames = _cu(np.stack([img, img]))

    def grab(f):
        r = sb.results()
        seg = r["seg_counts"][f].cpu().numpy()
        n = int(r["counts"][f].item())
        return {"n": n, "seg_counts": seg, "kpts": r["kpts"][f, :int(seg.sum())].cpu().numpy(),
                "orient": r["orient"][f, :int(seg.sum())].cpu().numpy(), "desc": r["desc"][f, :n].cpu().numpy(),
                "x": r["x"][f, :n].cpu().numpy(), "y": r["y"][f, :n].cpu().numpy()}

    for name in ("fov", "soft"):
        mask = g[f"{name}_mask"]
        sb.set_mask(mask if name == "fov" else _cu(mask))          # host and device mask images
        sb.run(frames)
        torch.cuda.synchronize()
        c = oracle.sift_frame(img, peak=0.0, want_levels=False, mask=mask)
        for f in range(2):
            p = grab(f)
            assert np.array_equal(p["seg_counts"], g[f"{name}_seg_counts"][: len(p["seg_counts"])]), name
            assert np.array_equal(p["kpts"], g[f"{name}_kpts"]), name
            assert_frame_matches(p, c, check_levels=False)
            relg = np.linalg.norm(p["desc"] - g[f"{name}_desc"], axis=1) / np.linalg.norm(g[f"{name}_desc"], axis=1)
            assert relg.max() <= 1e-3
    sb.set_mask(None)
    sb.run(frames)
    torch.cuda.synchronize()
    assert_frame_matches(grab(1), oracle.sift_frame(img, peak=0.0, want_levels=False), check_levels=False)
    sb.close()


def test_run_host_pipeline_equals_device_run(nm):
    """nm_sift_run_host splits a batch into stages of a few frames that run concurrently on several
    streams (H2D, kernels and D2H overlapped).  20 frames = 7 stages (each replayed as a CUDA graph on the second call): counts, descriptors and coordinates
    must be bitwise those of the single whole-batch nm_sift_run on device-resident frames."""
    n = 20
    frames = np.stack([synth.scene(256, 192, synth.SEED_BASE + (i % 5), shift=(0.5 * (i // 5), 0.25 * (i // 5)))
                       for i in range(n)])
    P = nm.SiftParams(256, 192)
    sb = nm.SiftBatch(P, n, 1024)
    sb.run(torch.from_numpy(frames).cuda())
    torch.cuda.synchronize()
    r = sb.results()
    counts = r["counts"].cpu().numpy().copy()
    desc = r["desc"].cpu().numpy().copy()
    xs = r["x"].cpu().numpy().copy()
    ys = r["y"].cpu().numpy().copy()
    for rep in range(2):                                   # second call reuses the cached stage descriptors
        out = sb.run_host(torch.from_numpy(frames).pin_memory())
        assert np.array_equal(out["counts"].numpy(), counts)
        assert counts.min() > 20
        for f in range(n):
            k = int(counts[f])
            assert np.array_equal(out["desc"][f, :k].numpy(), desc[f, :k]), (rep, f)
            assert np.array_equal(out["x"][f, :k].numpy(), xs[f, :k])
            assert np.array_equal(out["y"][f, :k].numpy(), ys[f, :k])
    sb.close()


def test_run_host_graphs_follow_the_context_state(nm):
    """The stage graphs of nm_sift_run_host are keyed by (frames, mask texture, descriptor mode): changing the mask or
    the descriptor mode between calls re-captures them, and the results equal the kernel-by-kernel nm_sift_run."""
    n, w, h = 12, 256, 192
    frames = np.stack([synth.scene(w, h, synth.SEED_BASE + 20 + i) for i in range(n)])
    yy, xx = np.mgrid[0:h, 0:w]
    mask = (((xx - w / 2) ** 2 + (yy - h / 2) ** 2) < (0.4 * h) ** 2).astype(np.float32)
    sb = nm.SiftBatch(nm.SiftParams(w, h), n, 2048)
    pinned = torch.from_numpy(frames).pin_memory()
    dev = torch.from_numpy(frames).cuda()

    def both():
        out = sb.run_host(pinned)
        c_host, d_host = out["counts"].numpy().copy(), out["desc"].numpy().copy()
        sb.run(dev)
        torch.cuda.synchronize()
        r = sb.results()
        c_dev, d_dev = r["counts"].cpu().numpy(), r["desc"].cpu().numpy()
        assert np.array_equal(c_host, c_dev)
        for f in range(n):
            assert np.array_equal(d_host[f, : c_dev[f]], d_dev[f, : c_dev[f]]), f
        return c_dev.copy()

    plain = both()
    sb.set_mask(mask)
    masked = both()
    assert (masked < plain).all() and (masked > 0).all()
    sb.set_exact_descriptor(True)
    both()
    sb.set_exact_descriptor(False)
    sb.set_mask(None)
    assert np.array_equal(both(), plain)
    sb.close()


def test_4k_six_octave_pyramid_and_extrema_vs_oracle(nm, oracle):
    """BASELINE.json configs[2]: 3840x2160, octave count forced to 6 (the default would be 7):
    Gaussian levels bitwise, keypoints bitwise, against the CPU oracle."""
    img = synth.scene(3840, 2160, synth.SEED_BASE + 3)
    c = oracle.sift_frame(img, peak=2.0, num_octaves=6, capacity=200000, want_levels=True, kp_cap=400000)
    P = nm.SiftParams(3840, 2160)
    P._num_octaves = 6
    P._peak_threshold = 2.0
    sb = nm.SiftBatch(P, 1, 65536)
    sb.run(_cu(img[None]))
    torch.cuda.synchronize()
    r = sb.results()
    n = int(r["counts"][0].item())
    assert c["n_oct"] == 6 and n == min(c["n"], 65536) and n > 1000
    for o in range(6):
        for l in range(6):
            assert np.array_equal(sb.level(0, o, l).cpu().numpy(), c["levels"][o][l]), (o, l)
    assert np.array_equal(r["seg_counts"][0].cpu().numpy(), c["seg_counts"])
    assert np.array_equal(r["kpts"][0, :n].cpu().numpy(), c["kpts"][:n])
    sb.close()


def test_stream_sharding_equals_single_run(nm):
    """BASELINE.json configs[4] at small scale: a stream of consecutive frames, SIFT + match(t -> t+1),
    sharded over 2 and 3 'ranks' (run one after the other here) with a one-frame overlap, must give
    exactly the single-rank result for every pair."""
    from niftymatch_b200.dist import match_stream
    n, w, h = 7, 320, 240
    frames = np.stack([synth.scene(w, h, synth.SEED_BASE + 9, shift=(0.75 * t, 0.5 * t)) for t in range(n)])
    fr = _cu(frames)
    P = nm.SiftParams(w, h)
    sb = nm.SiftBatch(P, 4, 4096)
    single = match_stream(sb, fr, 0.8, 1, 0, chunk=4)
    assert sorted(single) == list(range(n - 1))
    assert sum(int((m >= 0).sum()) for m in single.values()) > 50
    for world in (2, 3):
        merged = {}
        for rank in range(world):
            part = match_stream(sb, fr, 0.8, world, rank, chunk=3)
            assert not (set(part) & set(merged))
            merged.update(part)
        assert sorted(merged) == list(range(n - 1))
        for t in range(n - 1):
            assert torch.equal(merged[t], single[t]), (world, t)
    sb.close()


def test_gradient_arithmetic_is_bitwise_the_library_routines(nm):
    """The gradient kernels inline the main paths of the CUDA library's sqrtf / division / atan2f behind
    one range test (nm_gradient_from_diff).  It must agree bit for bit with the expression on the library
    routines (cudamath.cu:47-52) on every (dx, dy): 2^28 generated pairs (136 binades, image-scale
    magnitudes, quarter-integer pixel differences, zeros, subnormals, |dx| == |dy|, tiny vs large)."""
    import ctypes as C
    import niftymatch_b200._lib as L
    m = C.c_longlong(-1)
    assert L.load().nm_selftest_gradient(1 << 28, 12345, C.byref(m)) == 0
    assert m.value == 0
