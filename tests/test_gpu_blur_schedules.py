"""GPU suite, Gaussian pyramid: every blur kernel instantiation and every schedule of the streaming blur
(nm_pyramid.cu) against the CPU oracle, and the benchmark's own batch (64 x 1080p) through nm_sift_run and
nm_sift_run_host.

nm_blur_launch instantiates blur_tile_kernel<R, TMA>, blur_walk_kernel<R> and blur_strip_kernel<R> for R = 1..16 and
blur_stream_kernel<R, DST2> for R <= 13 (DST2: the launch also writes the decimated copy that becomes the next
octave's level 0), and picks the kernel and its schedule from the batch shape and the SM count.  The streaming kernel
runs either persistent (stream_min_ctas(R) CTAs per SM walking N full rounds of strips, then a split remainder) or
oversubscribed (P = 1..8 CTAs per strip).  Each case below runs once under torch.profiler and records the kernels and
grids it launched; test_blur_kernel_and_schedule_coverage asserts that the file as a whole ran every instantiation
and every schedule, so that a change to the heuristics that moves a case onto another path is reported instead of
leaving a kernel untested.

Batches are built on the device from 4 distinct scenes repeated: every frame must be bitwise the first frame of its
scene (this catches errors that depend on a frame's position in the launch anywhere in the batch), and the CPU checks
one or two frames per scene."""
import ctypes as C
import json
import os
import re
import tempfile
from collections import namedtuple

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

from niftymatch_b200 import synth  # noqa: E402
from tests._util import ang_diff, gray_double_formula  # noqa: E402
from tests.test_gpu_parity import DESC_REL_TOL, ORIENT_TOL, read_frame  # noqa: E402

SMS = 148                  # B200: the batch sizes below are chosen for this SM count
N_SCENES = 4
SEED = synth.SEED_BASE + 60


@pytest.fixture(scope="module")
def nm():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import niftymatch_b200 as nm
    nm.load()
    return nm


def _cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def stream_min_ctas(R):
    """Resident CTAs per SM of blur_stream_kernel<R> (nm_pyramid.cu)."""
    return 5 if R <= 10 else 4


# ------------------------------------------------------------------ inputs and references, computed once
_scene_cache, _oracle_cache = {}, {}


def _scenes(w, h):
    """(N_SCENES, h, w) float32 synthetic scenes."""
    if (w, h) not in _scene_cache:
        _scene_cache[(w, h)] = np.stack([synth.scene(w, h, SEED + i) for i in range(N_SCENES)])
    return _scene_cache[(w, h)]


def _bgra_scenes(w, h):
    """The scenes as BGRA frames whose three colour weights all matter (blue a shifted copy, red inverted)."""
    s = _scenes(w, h).astype(np.uint8)
    out = np.empty(s.shape + (4,), np.uint8)
    out[..., 0] = np.roll(s, 3, axis=2)
    out[..., 1] = s
    out[..., 2] = 255 - s // 2
    out[..., 3] = 255
    return out


def _oracle_frame(oracle, w, h, i, capacity):
    key = (w, h, i, capacity)
    if key not in _oracle_cache:
        _oracle_cache[key] = oracle.sift_frame(_scenes(w, h)[i], capacity=capacity)
    return _oracle_cache[key]


def _batch(scenes, n):
    """n frames on the device, frame f = scene f % len(scenes)."""
    idx = torch.arange(n, device="cuda") % len(scenes)
    return _cu(scenes)[idx].contiguous()


def _convolve(oracle, img, taps, R):
    img = np.ascontiguousarray(img, np.float32)
    h, w = img.shape
    res, buf = np.zeros_like(img), np.zeros_like(img)
    oracle.lib.orc_convolve(res.ctypes.data_as(C.c_void_p), img.ctypes.data_as(C.c_void_p), buf.ctypes.data_as(C.c_void_p),
                            w, h, taps.ctypes.data_as(C.c_void_p), R)
    return res


# ------------------------------------------------------------------ what ran: torch.profiler kernel events
Launch = namedtuple("Launch", "kernel R flag grid")
_KERNEL = re.compile(r"\b(blur_(?:tile|walk|strip|stream)_kernel)<(\d+)(?:,\s*([^>]+))?>")
_FLAGS = {"true": True, "1": True, "(bool)1": True, "false": False, "0": False, "(bool)0": False}

# case id -> [(launches of one traced run, column strips of its octave 0, radius of its base blur)]
_seen = {}


def _traced(case, fn, strips, base_radius=7):
    """Run fn() under torch.profiler (CUDA activity) and record the blur kernels it launched, in launch order, with
    their grids (kernel events of the exported trace carry "grid" and "block")."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    launches = []
    for e in sorted((e for e in events if e.get("cat") == "kernel"), key=lambda e: float(e["ts"])):
        m = _KERNEL.search(e.get("name", ""))
        if not m:
            continue
        grid = e.get("args", {}).get("grid")
        assert grid is not None, f"kernel event without a grid: {e}"
        flag = None if m.group(3) is None else _FLAGS[m.group(3).strip()]
        launches.append(Launch(m.group(1), int(m.group(2)), flag, tuple(int(g) for g in grid)))
    assert launches, "no blur kernel in the trace"
    _seen.setdefault(case, []).append((launches, strips, base_radius))
    return launches


def _schedule(launches, strips, base_radius):
    """What octave 0's base blur did, from the kernel and grid of the first launch at its radius: octave 0's level
    2 has the base blur's radius with the default sigmas and runs the same schedule, which matters because the trace
    of a 1080p run does not always contain the run's very first kernel.  Persistent launches have
    stream_min_ctas(R) x SMS CTAs, oversubscribed ones parts x strips."""
    launch = next(k for k in launches if k.R == base_radius)
    resident = stream_min_ctas(launch.R) * SMS
    if launch.kernel == "blur_stream_kernel":
        g = launch.grid[0]
        if g == resident:
            return f"persistent, {strips // resident} rounds"
        return f"parts = {g // strips}" if g % strips == 0 else f"blur_stream_kernel grid {g}"
    if launch.kernel == "blur_strip_kernel" and launch.R <= 13:
        return f"blur_strip_kernel at {strips // resident} rounds"
    return f"{launch.kernel}<{launch.R}>"


# ------------------------------------------------------------------ comparisons on the device
class _View:
    def __init__(self, ptr, shape, strides):
        self.__cuda_array_interface__ = {"shape": shape, "typestr": "<i4", "data": (ptr, False), "version": 2,
                                         "strides": strides}


def _octave_levels(sb, o, n):
    """The six Gaussian levels of octave o of frames 0..n-1 as one (n, 6, h, w) int32 view (bit patterns) of the
    workspace."""
    l0 = sb.level(0, o, 0)
    h, w = l0.shape
    lstride = sb.level(0, o, 1).data_ptr() - l0.data_ptr()
    fstride = sb.level(1, o, 0).data_ptr() - l0.data_ptr() if n > 1 else 6 * lstride
    return torch.as_tensor(_View(l0.data_ptr(), (n, 6, h, w), (fstride, lstride, 4 * l0.stride(0), 4)), device="cuda")


def _assert_scenes_repeat(sb, n):
    """Frame f of the last run (scene f % N_SCENES) is bitwise frame f % N_SCENES: every Gaussian level, the
    segment counts and, up to the frame's counts, keypoints, orientations, descriptors and coordinates."""
    k = N_SCENES
    for o in range(sb.n_oct):
        lv = _octave_levels(sb, o, n)
        for s in range(k):
            bad = (lv[s::k] != lv[s]).flatten(1).any(1)
            assert not bad.any(), f"octave {o}: frames {(s + k * torch.nonzero(bad)[:8, 0]).tolist()} differ from frame {s}"
    r = sb.results()
    counts, seg = r["counts"][:n], r["seg_counts"][:n]
    for s in range(k):
        assert (counts[s::k] == counts[s]).all() and (seg[s::k] == seg[s]).all(), s
        c = int(counts[s].item())
        nk = min(int(seg[s].sum().item()), sb.capacity)
        for key, m in (("kpts", nk), ("orient", nk), ("desc", c), ("x", c), ("y", c)):
            t = r[key][:n].view(torch.int32)
            assert (t[s::k, :m] == t[s, :m]).all(), (key, s)


def _assert_vs_oracle(p, c):
    """p: product frame (read_frame), c: oracle frame.  Levels, segment counts, counts, keypoints and descriptor
    coordinates bitwise.  Orientation histograms are reduced in a fixed lane order, the oracle's in raster order, and
    where a histogram peak is nearly flat the parabolic peak fit magnifies that last-bit difference (up to 4e-4 rad
    seen on these frames, about one keypoint in a thousand): orientations are held to ORIENT_TOL except for at most
    0.5 % of the keypoints, which must stay within the 1e-3 rad of BASELINE.json's north star.  Descriptors are held
    to DESC_REL_TOL wherever the orientations agree to ORIENT_TOL; the others are computed at another angle and are
    left out, as in smoke()."""
    assert np.array_equal(p["seg_counts"], c["seg_counts"]) and p["n"] == c["n"]
    for o in range(len(c["levels"])):
        for l in range(6):
            assert np.array_equal(p["levels"][o][l], c["levels"][o][l]), f"octave {o} level {l} not bitwise equal"
    assert np.array_equal(p["kpts"], c["kpts"]), "keypoints not bitwise equal"
    assert np.array_equal(p["orient"] < 0, c["orient"] < 0)
    d = np.where(c["orient"] >= 0, ang_diff(p["orient"], c["orient"]), 0.0)
    assert d.max() <= 1e-3 and (d > ORIENT_TOL).any(axis=1).mean() <= 5e-3, (d.max(), (d > ORIENT_TOL).sum())
    n = c["n"]
    if n:
        rel = np.linalg.norm(p["desc"] - c["desc"], axis=1) / np.maximum(np.linalg.norm(c["desc"], axis=1), 1e-20)
        same = (d[:n] <= ORIENT_TOL).all(axis=1)
        assert rel[same].max(initial=0.0) <= DESC_REL_TOL, rel[same].max(initial=0.0)
        assert np.array_equal(p["x"], c["x"]) and np.array_equal(p["y"], c["y"])


def _assert_same_frame(a, b, what):
    for key in ("n", "seg_counts", "kpts", "orient", "desc", "x", "y"):
        assert np.array_equal(a[key], b[key]), (what, key)
    for o in range(len(b["levels"])):
        for l in range(6):
            assert np.array_equal(a["levels"][o][l], b["levels"][o][l]), (what, o, l)


# ------------------------------------------------------------------ a. every radius through the pyramid
RADII = list(range(1, 17))


def _radius_case(nm, oracle, R):
    """64 frames of 640 x 480 with every blur of the pyramid at radius R (radius = ceil(4 sigma)).  With 148 SMs:
    octave 0 takes blur_stream_kernel<R, false> (persistent) and, for the level-3 blur that also writes octave 1's
    level 0, blur_stream_kernel<R, true> -- blur_strip_kernel<R> for R > 13; octave 1 (768 tiles) takes
    blur_walk_kernel<R>, octaves 2 and 3 blur_tile_kernel<R, true>.  The same frames as BGRA send the base blur
    through blur_strip_kernel<R> with the grey conversion fused, and must give bitwise the same results.
    The level sigmas alternate between the two ends of the interval of radius R, (R - 1) / 4 and R / 4: with five
    equal sigmas the DoG magnitude falls monotonically from level to level and no scale-space extremum exists, so the
    detector and everything after it would run on nothing."""
    w, h, n = 640, 480, 64
    big, small = R / 4.0, (R - 1) / 4.0 + 1 / 64
    taps = {}
    for sigma in (big, small):
        taps[sigma], radius = nm.gaussian_taps(sigma)
        assert radius == R
    sigmas = [small, big, small, big, small]
    P = nm.SiftParams(w, h)
    P._base_smooth = big
    for i in range(5):
        P.c.sigmas[i] = sigmas[i]
    bgra = _bgra_scenes(w, h)
    gray = gray_double_formula(bgra)
    sb = nm.SiftBatch(P, n, 4096)
    frames = _batch(gray, n)
    strips = -(-w // 128) * n
    _traced(f"radius {R}", lambda: sb.run(frames), strips, R)
    assert sb.results()["counts"][:n].sum() > 0, "no keypoints"
    _assert_scenes_repeat(sb, n)
    # each blur on its own against the oracle, on the first and the last frame
    for f in (0, n - 1):
        p = read_frame(sb, f)
        lv = p["levels"]
        assert np.array_equal(lv[0][0], _convolve(oracle, gray[f % N_SCENES], taps[big], R)), (f, 0, 0)
        for o in range(sb.n_oct):
            if o:
                oh, ow = lv[o][0].shape
                assert np.array_equal(lv[o][0], lv[o - 1][3][::2, ::2][:oh, :ow]), (f, o, 0)
            for l in range(5):
                assert np.array_equal(lv[o][l + 1], _convolve(oracle, lv[o][l], taps[sigmas[l]], R)), (f, o, l + 1)
    ref = [read_frame(sb, f) for f in range(N_SCENES)]
    del frames
    frames_bgra = _batch(bgra, n)
    _traced(f"radius {R}, BGRA", lambda: sb.run_bgra(frames_bgra), strips, R)
    _assert_scenes_repeat(sb, n)
    for f in range(N_SCENES):
        _assert_same_frame(read_frame(sb, f), ref[f], f"BGRA frame {f}")
    sb.close()
    del frames_bgra
    torch.cuda.empty_cache()


@pytest.mark.parametrize("R", RADII)
def test_pyramid_blur_radius_sweep(nm, oracle, R):
    _radius_case(nm, oracle, R)


# ------------------------------------------------------------------ b. every schedule of the streaming blur
# (schedule of octave 0's base blur with 148 SMs, frame width, height, batch); base blur R = 7, 740 resident CTAs.
# parts = P when P parts of >= 16 row groups bring 2 x strips x P to 3 x 740 (the smallest P reaching 5 x 740);
# persistent when no P qualifies: strips // 740 full rounds, the piece table holding up to 31 of them plus the split
# remainder -- one more round and the launch falls back to blur_strip_kernel.  parts = 2 is the benchmark's batch.
SCHEDULES = [
    ("parts = 1", 640, 480, 222),              # 1110 strips, 31 row groups: parts of 16 groups allow P = 1 only
    ("parts = 3", 256, 2048, 320),             # 129 row groups: P <= 8
    ("parts = 4", 256, 2048, 240),
    ("parts = 5", 256, 2048, 200),
    ("parts = 6", 256, 2048, 160),
    ("parts = 7", 256, 2048, 140),
    ("parts = 8", 256, 2048, 75),
    ("persistent, 2 rounds", 1920, 64, 100),   # 5 row groups: always persistent; 1500 strips
    ("persistent, 31 rounds", 1920, 64, 1530),  # 22950 strips: the last round count the 32-piece table holds
    ("blur_strip_kernel at 32 rounds", 1920, 64, 1579),
]
SCHEDULE_CAPACITY = 2048


def _schedule_case(nm, oracle, label, w, h, n):
    P = nm.SiftParams(w, h)
    sb = nm.SiftBatch(P, n, SCHEDULE_CAPACITY)
    frames = _batch(_scenes(w, h), n)
    _traced(label, lambda: sb.run(frames), -(-w // 128) * n)
    del frames
    _assert_scenes_repeat(sb, n)
    for s in range(N_SCENES):
        _assert_vs_oracle(read_frame(sb, s), _oracle_frame(oracle, w, h, s, SCHEDULE_CAPACITY))
    sb.close()
    torch.cuda.empty_cache()


@pytest.mark.parametrize("label,w,h,n", SCHEDULES, ids=["parts1", "parts3", "parts4", "parts5", "parts6", "parts7", "parts8",
                                                         "persistent2", "persistent31", "strip32"])
def test_stream_blur_schedule_vs_oracle(nm, oracle, label, w, h, n):
    """Default parameters: all levels, segment counts and keypoints bitwise the oracle's on each scene, descriptors
    within tolerance, and every frame of the batch bitwise the first frame of its scene."""
    _schedule_case(nm, oracle, label, w, h, n)


# ------------------------------------------------------------------ 3. the benchmark's batch
BENCH_N, BENCH_CAP = 64, 16384
RESULT_KEYS = ("counts", "seg_counts", "kpts", "orient", "desc", "x", "y")


@pytest.fixture(scope="module")
def bench_run(nm):
    """bench.py's headline step: frame g = synth.scene(1920, 1080, SEED_BASE + g), SiftBatch(P, 64, 16384), one
    nm_sift_run (octave 0 oversubscribed with 2 CTAs per strip, octaves 1.. on the side stream).  Results are kept
    on the host; the context stays open for the host-pipeline test."""
    frames = np.stack([synth.scene(1920, 1080, synth.SEED_BASE + g) for g in range(BENCH_N)])
    P = nm.SiftParams(1920, 1080)
    sb = nm.SiftBatch(P, BENCH_N, BENCH_CAP)
    dev = _cu(frames)
    _traced("benchmark batch", lambda: sb.run(dev), 15 * BENCH_N)
    res = {k: v.cpu().numpy().copy() for k, v in sb.results().items()}
    sampled = {f: read_frame(sb, f) for f in (0, BENCH_N // 2 - 1, BENCH_N - 1)}
    yield {"frames": frames, "dev": dev, "P": P, "sb": sb, "res": res, "sampled": sampled}
    sb.close()
    del dev
    torch.cuda.empty_cache()


def _assert_frame_results_equal(got, g, ref, f, keys, what):
    """Frame g of `got` bitwise frame f of `ref` (host arrays indexed [frame, ...]), up to the frame's counts."""
    c = int(ref["counts"][f])
    nk = min(int(ref["seg_counts"][f].sum()), BENCH_CAP)
    assert got["counts"][g] == c, (what, f)
    for key in keys:
        m = {"seg_counts": None, "kpts": nk, "orient": nk}.get(key, c)
        assert np.array_equal(got[key][g, :m], ref[key][f, :m]), (what, f, key)


def test_benchmark_batch_vs_oracle(bench_run, oracle):
    res = bench_run["res"]
    assert (res["counts"] > 5000).all()
    for f, p in bench_run["sampled"].items():
        _assert_vs_oracle(p, oracle.sift_frame(bench_run["frames"][f], capacity=BENCH_CAP))


def test_benchmark_batch_in_eight_calls(nm, bench_run):
    """The same frames as 8 calls of 8 frames (octave 0 on the tile-walking blur: 2040 tiles but fewer strip chunks
    than the strip kernels take; no side stream): every result bitwise."""
    ref = bench_run["res"]
    sb = nm.SiftBatch(bench_run["P"], 8, BENCH_CAP)
    for k in range(BENCH_N // 8):
        part = bench_run["dev"][8 * k: 8 * k + 8]
        if k == 0:
            _traced("benchmark frames, 8 per call", lambda: sb.run(part), 15 * 8)
        else:
            sb.run(part)
            torch.cuda.synchronize()
        got = {key: v.cpu().numpy() for key, v in sb.results().items()}
        for i in range(8):
            _assert_frame_results_equal(got, i, ref, 8 * k + i, RESULT_KEYS[1:], "8 x 8")
    sb.close()


def test_benchmark_batch_through_run_host(bench_run):
    """nm_sift_run_host on the pinned 64 frames (3-frame stages, tapered end, four streams): the first call captures
    the stage graphs, the second replays them.  Counts, descriptors and coordinates bitwise the device run's."""
    ref, sb = bench_run["res"], bench_run["sb"]
    pinned = torch.from_numpy(bench_run["frames"]).pin_memory()
    out = None
    for call in ("capture", "replay"):
        out = sb.run_host(pinned, out=out)
        got = {k: v.numpy() for k, v in out.items()}
        assert np.array_equal(got["counts"], ref["counts"]), call
        for f in range(BENCH_N):
            _assert_frame_results_equal(got, f, ref, f, ("desc", "x", "y"), call)


# ------------------------------------------------------------------ c. coverage, from what ran
def test_blur_kernel_and_schedule_coverage(nm, oracle, bench_run, capsys):
    """The union of the traced runs of this file contains every blur kernel instantiation and every schedule of
    octave 0's base blur listed in SCHEDULES (plus parts = 2 from the benchmark batch).  Cases that did not run in
    this session (a -k selection) are run here."""
    if torch.cuda.get_device_properties(0).multi_processor_count != SMS:
        pytest.skip(f"kernel and schedule choices are sized for {SMS} SMs")
    for R in RADII:
        if f"radius {R}" not in _seen:
            _radius_case(nm, oracle, R)
    for case in SCHEDULES:
        if case[0] not in _seen:
            _schedule_case(nm, oracle, *case)
    ran = set()
    schedules = {}
    for case, runs in _seen.items():
        for launches, strips, base_radius in runs:
            ran |= {(k.kernel, k.R, k.flag) for k in launches}
            schedules.setdefault(_schedule(launches, strips, base_radius), []).append(case)
    need = {("blur_stream_kernel", R, d) for R in range(1, 14) for d in (False, True)}
    need |= {(k, R, None) for k in ("blur_walk_kernel", "blur_strip_kernel") for R in RADII}
    need |= {("blur_tile_kernel", R, True) for R in RADII}
    missing = sorted(need - ran, key=str)
    assert not missing, f"kernel instantiations no case launched: {missing}"
    need_sched = {s[0] for s in SCHEDULES} | {"parts = 2"}
    missing = sorted(need_sched - set(schedules))
    assert not missing, f"schedules no case ran: {missing}; base-blur schedules seen: {schedules}"
    with capsys.disabled():
        print(f"\nblur kernels launched ({len(ran)}):", sorted(ran, key=str))
        for s, cases in sorted(schedules.items()):
            print(f"octave-0 base blur {s}: {cases}")
