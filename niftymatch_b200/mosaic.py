"""Mosaic of a registered frame stream through the C-ABI (nm_mosaic_*): the pairwise homographies chained and laid
out on a canvas (place), a chunk of BGRA frames blended in one pass over the canvas (Mosaic.blend), and the two
together for a whole stream (render_stream).  Torch tensors as device memory."""
from __future__ import annotations

import ctypes as C
from collections import namedtuple

import numpy as np

from . import _lib
from ._lib import check
from .sift import _stream_ptr

# Device tensors written by nm_mosaic_place_f32: mats (n, 9) float32 canvas-local -> frame matrices, rects (n, 4)
# int32 (tx, ty, nw, nh) in canvas pixels, flags (n,) int32 (bit 0: pair replaced by the identity, bit 1: no
# footprint), bounds (4,) int32 (ox, oy, width, height), chain (n, 9) float64 frame -> mosaic transforms.
Placement = namedtuple("Placement", "mats rects flags bounds chain")


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _dev(a, dtype):
    import torch
    if isinstance(a, torch.Tensor):
        return a.to(device="cuda", dtype=dtype).contiguous()
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype, device="cuda")


def place(H, status, frame_w: int, frame_h: int, anchor=None, origin=None) -> Placement:
    """Placement of n = len(H) + 1 frames.  H: (n-1, 9) pairwise homographies, H[p] maps frame p to frame p+1 (the
    nm_ransac_batch_f32 convention); status: (n-1, 3) as that call writes it, or None.  anchor: 9 floats, frame 0 ->
    mosaic (default identity); origin: (ox, oy) of a fixed canvas (default: fitted to the footprints).  Asynchronous."""
    import torch
    H = _dev(H, torch.float32).reshape(-1, 9)
    n = H.shape[0] + 1
    st = _dev(status, torch.int32).reshape(-1, 3) if status is not None else None
    assert st is None or st.shape[0] == n - 1
    an = _dev(anchor, torch.float32).reshape(9) if anchor is not None else None
    org = _dev(origin, torch.int32).reshape(2) if origin is not None else None
    out = Placement(torch.empty((n, 9), dtype=torch.float32, device="cuda"), torch.empty((n, 4), dtype=torch.int32, device="cuda"),
                    torch.empty(n, dtype=torch.int32, device="cuda"), torch.empty(4, dtype=torch.int32, device="cuda"),
                    torch.empty((n, 9), dtype=torch.float64, device="cuda"))
    check(_lib.load().nm_mosaic_place_f32(_p(H) if n > 1 else None, _p(st), n, frame_w, frame_h, _p(an), _p(org), _p(out.mats),
                                          _p(out.rects), _p(out.flags), _p(out.bounds), _p(out.chain), _stream_ptr()),
          "nm_mosaic_place_f32")
    return out


class Mosaic:
    """Frame-slot textures of one frame size (nm_mosaic_create).  mask: (frame_h, frame_w) uint8, weights:
    (frame_h, frame_w) float32, numpy or torch, host or device."""

    def __init__(self, frame_w: int, frame_h: int, max_frames: int, mask, weights):
        import torch
        self.lib = _lib.load()
        self.fw, self.fh, self.max_frames = frame_w, frame_h, max_frames
        mask = mask.contiguous() if isinstance(mask, torch.Tensor) else np.ascontiguousarray(mask, dtype=np.uint8)
        weights = weights.contiguous() if isinstance(weights, torch.Tensor) else np.ascontiguousarray(weights, dtype=np.float32)
        assert tuple(mask.shape) == (frame_h, frame_w) and tuple(weights.shape) == (frame_h, frame_w)
        assert mask.dtype in (np.uint8, torch.uint8) and weights.dtype in (np.float32, torch.float32)
        ptr = lambda a: C.c_void_p(a.data_ptr() if isinstance(a, torch.Tensor) else a.ctypes.data)
        self._ctx = C.c_void_p()
        check(self.lib.nm_mosaic_create(C.byref(self._ctx), frame_w, frame_h, max_frames, ptr(mask), ptr(weights)), "nm_mosaic_create")

    def close(self):
        if self._ctx:
            self.lib.nm_mosaic_destroy(self._ctx)
            self._ctx = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def place(self, H, status=None, anchor=None, origin=None) -> Placement:
        return place(H, status, self.fw, self.fh, anchor, origin)

    def blend(self, frames_bgra, mats, rects, canvas, canvas_wts) -> None:
        """Blend frames_bgra (n, frame_h, frame_w, 4) uint8 cuda, n <= max_frames, into canvas (ch, cw, 4) uint8 and
        canvas_wts (ch, cw) float32 in place: bitwise n transform_blend calls in frame order.  Asynchronous."""
        import torch
        assert frames_bgra.is_cuda and frames_bgra.dtype == torch.uint8 and frames_bgra.is_contiguous()
        assert frames_bgra.dim() == 4 and frames_bgra.shape[-1] == 4
        assert canvas.dtype == torch.uint8 and canvas.is_contiguous() and canvas_wts.dtype == torch.float32 and canvas_wts.is_contiguous()
        ch, cw = canvas.shape[:2]
        assert tuple(canvas.shape) == (ch, cw, 4) and tuple(canvas_wts.shape) == (ch, cw)
        n = frames_bgra.shape[0]
        assert mats.shape[0] >= n and rects.shape[0] >= n and mats.is_contiguous() and rects.is_contiguous()
        check(self.lib.nm_mosaic_blend_bgra(self._ctx, _p(frames_bgra), n, frames_bgra.shape[2], frames_bgra.shape[1], _p(mats),
                                            _p(rects), _p(canvas), cw, ch, _p(canvas_wts), _stream_ptr()), "nm_mosaic_blend_bgra")

    def textures(self):
        """(frame slot textures [max_frames], mask texture, weight texture) as cudaTextureObject_t integers."""
        tex = (C.c_ulonglong * self.max_frames)()
        m, w = C.c_ulonglong(), C.c_ulonglong()
        check(self.lib.nm_mosaic_textures(self._ctx, tex, C.byref(m), C.byref(w)), "nm_mosaic_textures")
        return list(tex), m.value, w.value


def render_stream(frames_bgra, H, status, mask=None, weights=None, max_frames: int = 64, anchor=None, origin=None, mosaic=None):
    """The mosaic of a registered stream: place, ONE synchronisation to read the canvas size, then the frames blended in
    chunks of max_frames (or of mosaic.max_frames when a Mosaic is given instead of mask / weights).
    frames_bgra: (n, h, w, 4) uint8 cuda; H, status: the n - 1 pairs (nm_ransac_batch_f32).
    Returns (canvas (height, width, 4) uint8, canvas_wts (height, width) float32, Placement)."""
    import torch
    n, fh, fw = frames_bgra.shape[:3]
    own = mosaic is None
    if own:
        mosaic = Mosaic(fw, fh, min(max_frames, n), mask, weights)
    try:
        pl = place(H, status, fw, fh, anchor, origin)
        ox, oy, cw, ch = pl.bounds.tolist()
        canvas = torch.zeros((ch, cw, 4), dtype=torch.uint8, device=frames_bgra.device)
        cwts = torch.zeros((ch, cw), dtype=torch.float32, device=frames_bgra.device)
        if cw > 0 and ch > 0:
            for c0 in range(0, n, mosaic.max_frames):
                c1 = min(n, c0 + mosaic.max_frames)
                mosaic.blend(frames_bgra[c0:c1].contiguous(), pl.mats[c0:c1], pl.rects[c0:c1], canvas, cwts)
    finally:
        if own:
            torch.cuda.current_stream().synchronize()     # the enqueued blends read the context's frame slots
            mosaic.close()
    return canvas, cwts, pl
