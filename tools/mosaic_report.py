"""Mosaic of a frame stream on one GPU (nm_mosaic_*): 256 BGRA 1080p frames along a synthetic camera path, blended
in chunks of 64.  Reports the GPU and its power limit, the canvas, CUDA-event times in alternating windows of
  (a) the per-frame loop: one nm_transform_blend_bgra per frame on the context's textures (frames already in the slots),
  (b) nm_mosaic_blend_bgra, one call per chunk, including its copies of the frames into the slot arrays,
  (c) nm_mosaic_place_f32,
ms per frame, achieved GB/s against the measured 6 450.9 GB/s copy peak, and whether (a) and (b) give bitwise the same
canvas.  Algorithmic bytes come from the rects: 9 B per frame pixel (frame 4 + mask 1 + weights 4) plus 16 B (canvas
pixel and weight, read and written) per rect pixel for the loop, per touched canvas pixel for the one-pass blend.
The camera path is given as homographies (no SIFT): per frame 6 - 12 px of translation, 0.2 degrees of rotation and
0.2 % of scale.

    python tools/mosaic_report.py [--frames 256] [--chunk 64] [--windows 5] [--reps 3] [--lib other/libnm_b200.so]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

PEAK_GBS = 6450.9          # measured device-to-device copy peak of the B200 (DESIGN.md §4.5)


def camera_path(n, fw, fh, seed=7):
    """n - 1 pairwise homographies (frame p -> frame p + 1): a heading that turns slowly, 6 - 12 px per frame,
    +-0.2 degrees of rotation and +-0.2 % of scale about the frame centre."""
    rng = np.random.default_rng(seed)
    cx, cy = (fw - 1) / 2, (fh - 1) / 2
    T = lambda x, y: np.array([[1, 0, x], [0, 1, y], [0, 0, 1.0]])
    H, phi = [], 0.0
    for _ in range(n - 1):
        phi += rng.normal(0, 0.08)
        a = np.deg2rad(0.2 * rng.choice([-1, 1]))
        s = 1 + 0.002 * rng.choice([-1, 1])
        d = rng.uniform(6, 12)
        M = np.array([[s * np.cos(a), -s * np.sin(a), 0], [s * np.sin(a), s * np.cos(a), 0], [0, 0, 1.0]])
        H.append(T(cx + d * np.cos(phi), cy + d * np.sin(phi)) @ M @ T(-cx, -cy))
    return np.array(H, np.float32).reshape(-1, 9)


def fov_mask(fw, fh):
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float64)
    r = 0.49 * min(fw, fh)
    return ((((xx - (fw - 1) / 2) ** 2 + (yy - (fh - 1) / 2) ** 2) < r * r) * 255).astype(np.uint8)


def radial_weights(fw, fh):
    yy, xx = np.mgrid[0:fh, 0:fw].astype(np.float64)
    d = np.sqrt((xx - (fw - 1) / 2) ** 2 + (yy - (fh - 1) / 2) ** 2) / (0.5 * np.hypot(fw, fh))
    return np.ascontiguousarray(np.maximum(1.0 - d, 0.0) + 1.0 / 64, dtype=np.float32)


def gpu_identity(torch):
    name, limit = torch.cuda.get_device_name(0), "unknown"
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
        if out:
            name, limit = [s.strip() for s in out.split(",")[:2]]
    except (OSError, subprocess.SubprocessError):
        pass
    return name, limit


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--chunk", type=int, default=64)
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--scenes", type=int, default=4, help="distinct synth scenes the frames cycle through")
    ap.add_argument("--windows", type=int, default=5, help="alternating windows of (a), (b), (c)")
    ap.add_argument("--reps", type=int, default=3, help="timed renders per leg and window")
    ap.add_argument("--lib", default=None, help="another build of libnm_b200.so to measure (A/B of kernel variants)")
    a = ap.parse_args()

    import torch
    import niftymatch_b200._lib as L
    if a.lib:
        L.LIB_PATH = os.path.abspath(a.lib)
    import niftymatch_b200 as nm
    from niftymatch_b200 import synth
    assert torch.cuda.is_available(), "needs a CUDA device"
    lib = nm.load()
    n, fw, fh, chunk = a.frames, a.width, a.height, a.chunk
    name, limit = gpu_identity(torch)

    scenes = np.stack([np.rint(synth.scene(fw, fh, synth.SEED_BASE + s)).astype(np.uint8) for s in range(a.scenes)])
    grey = torch.from_numpy(scenes).cuda()[torch.arange(n) % a.scenes]
    frames = torch.empty((n, fh, fw, 4), dtype=torch.uint8, device="cuda")
    frames[..., :3] = grey[..., None]
    frames[..., 3] = 255
    del grey
    H = torch.from_numpy(camera_path(n, fw, fh)).cuda()
    mask, wts = fov_mask(fw, fh), radial_weights(fw, fh)
    fused = nm.Mosaic(fw, fh, chunk, mask, wts)
    every = nm.Mosaic(fw, fh, n, mask, wts)          # the per-frame loop reads frame k from slot k
    pl = nm.place(H, None, fw, fh)
    ox, oy, cw, ch = pl.bounds.tolist()
    rects = pl.rects.cpu().numpy()
    assert (pl.flags.cpu().numpy() == 0).all()
    canvas = torch.zeros((ch, cw, 4), dtype=torch.uint8, device="cuda")
    cwts = torch.zeros((ch, cw), dtype=torch.float32, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    tex, mtex, wtex = every.textures()
    mats_p = pl.mats.data_ptr()
    every.blend(frames, pl.mats, pl.rects, canvas, cwts)              # fills every slot

    def loop():
        for k in range(n):
            tx, ty, nw, nh = (int(v) for v in rects[k])
            rc = lib.nm_transform_blend_bgra(C.c_void_p(canvas.data_ptr()), cw, ch, tex[k], fw, fh, nw, nh, C.c_void_p(mats_p + 36 * k),
                                             tx, ty, mtex, C.c_void_p(cwts.data_ptr()), wtex, stream)
            assert rc == 0

    def one_pass():
        for c0 in range(0, n, chunk):
            c1 = min(n, c0 + chunk)
            fused.blend(frames[c0:c1], pl.mats[c0:c1], pl.rects[c0:c1], canvas, cwts)

    def placement():
        nm.place(H, None, fw, fh)

    legs = {"a_per_frame_loop": loop, "b_one_pass": one_pass, "c_place": placement}
    # bitwise check at the timed size, and warm-up of every leg
    results = {}
    for k in ("a_per_frame_loop", "b_one_pass"):
        canvas.zero_()
        cwts.zero_()
        legs[k]()
        torch.cuda.synchronize()
        results[k] = (canvas.clone(), cwts.clone())
    placement()
    bitwise = torch.equal(results["a_per_frame_loop"][0], results["b_one_pass"][0]) and \
        torch.equal(results["a_per_frame_loop"][1].view(torch.int32), results["b_one_pass"][1].view(torch.int32))
    covered = int((results["b_one_pass"][1] > 0).sum())
    del results

    times = {k: [] for k in legs}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(a.windows):
        for k, fn in legs.items():
            for _ in range(a.reps):
                canvas.zero_()
                cwts.zero_()
                ev[0].record()
                fn()
                ev[1].record()
                ev[1].synchronize()
                times[k].append(ev[0].elapsed_time(ev[1]))

    # algorithmic bytes from the rects (all of them lie inside the fitted canvas)
    cover = torch.zeros((ch, cw), dtype=torch.int32, device="cuda")
    for tx, ty, nw, nh in rects:
        cover[ty: ty + nh, tx: tx + nw] += 1
    touched = int((cover > 0).sum())
    rect_px = int((rects[:, 2].astype(np.int64) * rects[:, 3]).sum())
    frame_px = n * fw * fh
    bytes_loop = 9 * frame_px + 16 * rect_px
    bytes_fused = 9 * frame_px + 16 * touched
    med = {k: float(np.median(v)) for k, v in times.items()}
    out = {
        "gpu": name, "power_limit": limit, "frames": n, "frame": [fw, fh], "chunk": chunk, "canvas": [cw, ch],
        "origin": [ox, oy], "rect_area_sum_px": rect_px, "touched_canvas_px": touched, "blended_canvas_px": covered,
        "ms": {k: {"median": round(med[k], 3), "min": round(min(v), 3), "max": round(max(v), 3)} for k, v in times.items()},
        "ms_per_frame": {k: round(med[k] / n, 4) for k in ("a_per_frame_loop", "b_one_pass")},
        "algorithmic_bytes": {"a_per_frame_loop": bytes_loop, "b_one_pass": bytes_fused},
        "gbs": {"a_per_frame_loop": round(bytes_loop / med["a_per_frame_loop"] / 1e6, 1),
                "b_one_pass": round(bytes_fused / med["b_one_pass"] / 1e6, 1)},
        "fraction_of_copy_peak": {"a_per_frame_loop": round(bytes_loop / med["a_per_frame_loop"] / 1e6 / PEAK_GBS, 3),
                                  "b_one_pass": round(bytes_fused / med["b_one_pass"] / 1e6 / PEAK_GBS, 3)},
        "speedup_b_over_a": round(med["a_per_frame_loop"] / med["b_one_pass"], 3),
        "bitwise_equal_a_b": bool(bitwise),
        "windows": a.windows, "reps": a.reps, "lib": L.LIB_PATH,
    }
    print(f"{name}, power limit {limit}")
    print(f"{n} frames {fw}x{fh} in chunks of {chunk}; canvas {cw}x{ch} at ({ox}, {oy}); sum of rect areas {rect_px / 1e6:.1f} Mpx, "
          f"touched canvas {touched / 1e6:.2f} Mpx")
    for k in legs:
        extra = f", {med[k] / n:.4f} ms/frame, {out['gbs'][k]} GB/s ({out['fraction_of_copy_peak'][k]} of {PEAK_GBS})" if k in out["gbs"] else ""
        print(f"  {k}: median {med[k]:.3f} ms (min {min(times[k]):.3f}, max {max(times[k]):.3f}){extra}")
    print(f"  (b) over (a): {out['speedup_b_over_a']}x; canvases bitwise equal: {bitwise}")
    print(json.dumps(out))
    fused.close()
    every.close()
    return 0 if bitwise else 1


if __name__ == "__main__":
    sys.exit(main())
